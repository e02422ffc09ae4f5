"""Cost of teacher-forced scoring: ``model.score`` (fc_out with the log-sum-exp epilogue, no logits) against today's
route, ``model.decoder`` + ``torch.log_softmax`` + ``gather`` (three fp32 [B, T, V] tensors), from encoder output at
B = 1, 8, 64, 256 and T = 40, 150; ``score`` from images at B = 256, T = 150 with greedy ``generate`` at the same
shape for context.  One process; the forms of a shape are alternated call by call and each call is timed with CUDA
events; every shape is warmed up first.  Each route runs on its own engine, so each workspace holds only that route's
buffers; the peak allocation of a route is its workspace plus the largest allocation above it during one call.

    python profiles/score_bench.py [--calls 20] [--out profiles/score_bench.json]
    python profiles/score_bench.py --profile [--out DIR/score_phases.json]     # per-phase kernel times, torch.profiler

The synthetic checkpoint never emits eos, so every position is scored and greedy decodes all T steps.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from handwritten_math_ocr_api_b200 import FormulaRecognitionModel  # noqa: E402
from handwritten_math_ocr_api_b200.layout import ModelConfig  # noqa: E402
from handwritten_math_ocr_api_b200.synthetic import synth_images, synth_state_dict  # noqa: E402

SHAPES = [(b, t) for t in (40, 150) for b in (1, 8, 64, 256)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def timed(f):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    f()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def peak_bytes(model, f):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    f()
    torch.cuda.synchronize()
    return model.workspace_bytes() + torch.cuda.max_memory_allocated() - base


def stats(v, batch):
    med = statistics.median(v)
    return {"median_ms": med, "min_ms": min(v), "max_ms": max(v), "images_per_s": batch / med * 1e3}


def inputs(V, B, T, seed):
    g = torch.Generator().manual_seed(seed)
    feats = torch.randn(B, 30, 256, generator=g).cuda()
    tok = torch.randint(3, V, (B, T + 1), generator=g).cuda()
    tok[:, 0] = 1
    return feats, tok


def torch_route(m, feats, tok):
    logits = m.decoder(feats, tok[:, :-1])
    return torch.log_softmax(logits, -1).gather(-1, tok[:, 1:].unsqueeze(-1)).squeeze(-1)


def bench(a, sd, cfg):
    V = cfg.vocab_size
    m_score, m_torch, m_gen = (FormulaRecognitionModel(V) for _ in range(3))
    for m in (m_score, m_torch, m_gen):
        m.load_state_dict(sd)
    res = {"gpu": gpu_info(), "calls": a.calls, "vocab": V, "weights": "synthetic seed 0, eos never emitted",
           "timing": "CUDA events around each call, forms alternated call by call, after 3 warm-up calls per form",
           "encoder_output": []}
    for B, T in SHAPES:
        feats, tok = inputs(V, B, T, seed=B * 1000 + T)
        forms = {"score": (m_score, lambda: m_score.score(encoder_out=feats, tokens=tok)),
                 "decoder_log_softmax_gather": (m_torch, lambda: torch_route(m_torch, feats, tok))}
        for _, f in forms.values():
            for _ in range(3):
                f()
        ms = {k: [] for k in forms}
        for _ in range(a.calls):
            for k, (_, f) in forms.items():
                ms[k].append(timed(f))
        row = {"batch": B, "T": T}
        for k, (m, f) in forms.items():
            row[k] = stats(ms[k], B)
            row[k]["peak_bytes"] = peak_bytes(m, f)
        row["speedup"] = row["decoder_log_softmax_gather"]["median_ms"] / row["score"]["median_ms"]
        print(json.dumps(row), flush=True)
        res["encoder_output"].append(row)
        del feats, tok
        torch.cuda.empty_cache()
    B, T = 256, 150
    imgs = synth_images(8, seed=1234).cuda().repeat(B // 8, 1, 1, 1).contiguous()
    _, tok = inputs(V, B, T, seed=7)
    forms = {"score_from_images": lambda: m_score.score(imgs, tokens=tok),
             "generate_greedy": lambda: m_gen.generate(imgs, max_len=T)}
    for f in forms.values():
        for _ in range(3):
            f()
    ms = {k: [] for k in forms}
    for _ in range(a.calls):
        for k, f in forms.items():
            ms[k].append(timed(f))
    res["images"] = {"batch": B, "T": T, **{k: stats(v, B) for k, v in ms.items()}}
    print(json.dumps(res["images"]), flush=True)
    return res


PHASES = [("projection_lse_epilogue", lambda n: "gemm_tcgen05_kernel<256, false, true>" in n),
          ("combine", lambda n: "score_combine" in n),
          ("prefill_self_attention", lambda n: "prefill_self" in n),
          ("decoder_layers", lambda n: "hmocr" in n),
          ("torch_id_checks_and_other", lambda n: True)]


def profile(a, sd, cfg):
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile as tprofile
    V = cfg.vocab_size
    m = FormulaRecognitionModel(V)
    m.load_state_dict(sd)
    B, T = a.profile_batch, a.profile_t
    feats, tok = inputs(V, B, T, seed=3)
    for _ in range(3):
        m.score(encoder_out=feats, tokens=tok)
    torch.cuda.synchronize()
    with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(a.calls):
            m.score(encoder_out=feats, tokens=tok)
        torch.cuda.synchronize()
    per = {name: 0.0 for name, _ in PHASES}
    kernels = {}
    for ev in prof.key_averages():
        us = ev.self_device_time_total
        if ev.device_type != DeviceType.CUDA or us <= 0:
            continue
        kernels[ev.key] = us / a.calls / 1e3
        for name, match in PHASES:
            if match(ev.key):
                per[name] += us / a.calls / 1e3
                break
    total = sum(per.values())
    res = {"gpu": gpu_info(), "batch": B, "T": T, "calls": a.calls,
           "phase_ms_per_call": per, "phase_share": {k: v / total for k, v in per.items()},
           "kernel_ms_per_call": dict(sorted(kernels.items(), key=lambda kv: -kv[1]))}
    print(json.dumps(res, indent=1), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20, help="timed calls of each form and shape")
    ap.add_argument("--profile", action="store_true", help="per-phase kernel times of one score shape instead")
    ap.add_argument("--profile-batch", type=int, default=256)
    ap.add_argument("--profile-t", type=int, default=150)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    cfg = ModelConfig()
    sd = synth_state_dict(cfg, seed=0, eos_bias_sigma=0.0)
    res = profile(a, sd, cfg) if a.profile else bench(a, sd, cfg)
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
