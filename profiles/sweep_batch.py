"""Decode/encoder time of one generate() call as a function of the batch (latency- vs throughput-bound check).

"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from handwritten_math_ocr_api_b200 import FormulaRecognitionModel  # noqa: E402
from handwritten_math_ocr_api_b200.layout import ModelConfig  # noqa: E402
from handwritten_math_ocr_api_b200.synthetic import synth_images, synth_state_dict  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--batches", default="64,128,256,512")
ap.add_argument("--max-len", type=int, default=150)
ap.add_argument("--spl", type=int, default=0, help="steps per persistent-kernel launch (0 = engine default)")
a = ap.parse_args()
cfg = ModelConfig()
m = FormulaRecognitionModel(cfg.vocab_size)
m.load_state_dict(synth_state_dict(cfg, seed=0, eos_bias_sigma=0.0))
if a.spl:
    m.set_option("steps_per_launch", a.spl)
base = synth_images(8, seed=1234).cuda()
for B in [int(x) for x in a.batches.split(",")]:
    imgs = base.repeat((B + 7) // 8, 1, 1, 1)[:B].contiguous()
    for _ in range(3):
        m.generate(imgs, max_len=a.max_len)
    torch.cuda.synchronize()
    enc, dec = [], []
    for _ in range(3):
        m.generate(imgs, max_len=a.max_len)
        e, d = m.last_timings_ms()
        enc.append(e); dec.append(d)
    e, d = min(enc), min(dec)
    print(f"B={B:4d}: encoder {e:7.3f} ms  decode {d:7.3f} ms  ({d / a.max_len * 1e3:6.1f} us/step)  "
          f"{B / (e + d) * 1e3:8.1f} img/s", flush=True)
