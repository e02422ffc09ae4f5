"""Phase-by-phase latency breakdown of one decode step of the persistent cluster kernel
(clock64 stamps of cluster 0 / CTA 0 / thread 0; see hmocr_read_trace).

    python profiles/trace_step.py [--batch 240] [--step 100]
"""
import argparse
import ctypes as C
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from handwritten_math_ocr_api_b200 import FormulaRecognitionModel, _lib  # noqa: E402
from handwritten_math_ocr_api_b200.layout import ModelConfig  # noqa: E402
from handwritten_math_ocr_api_b200.synthetic import synth_images, synth_state_dict  # noqa: E402

LAYER = ["qkv: wait for the weight chunk", "qkv: 16 mma + epilogue + K issue", "qkv: block barrier", "self-attn: K/V blocks, online softmax, P.V", "self-attn: context send + append + prefetch", "wait context 1", "out-proj 1 tiles + y send", "wait y 1",
         "layernorm 1 + sync", "cross-q tiles + sync", "cross-attention + context send", "wait context 2",
         "out-proj 2 tiles + y send", "wait y 2", "layernorm 2 + sync", "linear1 tiles + hidden send", "wait hidden",
         "linear2 tiles + y send", "wait y 3", "layernorm 3 + sync", "next layer: bias wait"]
TAIL = ["fc_out tiles + warp reduce + sync", "partials send + wait", "token select + embed next + sync"]

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--step", type=int, default=100)
a = ap.parse_args()
cfg = ModelConfig()
m = FormulaRecognitionModel(cfg.vocab_size)
m.load_state_dict(synth_state_dict(cfg, seed=0, eos_bias_sigma=0.0))
imgs = synth_images(8, seed=1234).cuda()
imgs = imgs.repeat((a.batch + 7) // 8, 1, 1, 1)[: a.batch].contiguous()
enc = m.encoder(imgs)
m.generate(encoder_out=enc, max_len=150)
m.set_option("trace_step", a.step)
m.generate(encoder_out=enc, max_len=150)
torch.cuda.synchronize()
buf = (C.c_int64 * 1024)()
_lib.check(_lib.load().hmocr_read_trace(m._eng.handle, buf, 1024), "read_trace")
st = [x for x in buf if x != 0]
n_layer = len(LAYER)
L = cfg.num_layers
d = [st[i + 1] - st[i] for i in range(len(st) - 1)]
clk = 1.965e3    # cycles per us at max clock (approximate)
agg = {}
for l in range(L):
    base = l * n_layer
    for k, name in enumerate(LAYER):
        agg.setdefault(name, []).append(d[base + k])
print(f"B={a.batch} step {a.step}: {len(st)} stamps, step total {(st[-1]-st[0])/clk:.1f} us (at 1965 MHz)")
print("per-layer phases (mean over 8 layers, cycles -> us):")
tot = 0
for name in LAYER:
    v = sum(agg[name]) / len(agg[name])
    tot += v
    print(f"  {name:42s} {v:8.0f} cyc {v/clk:6.2f} us")
print(f"  {'layer total':42s} {tot:8.0f} cyc {tot/clk:6.2f} us")
base = L * n_layer
for k, name in enumerate(TAIL):
    if base + k < len(d):
        print(f"  {name:58s} {d[base+k]:8.0f} cyc {d[base+k]/clk:6.2f} us")
