"""Cost of the n-best outputs: generate(beam_size=5) against generate_nbest(beam_size=5, n_best=5), alternated in one
process, B = 64, T = 150, the checkpoint that never emits eos (every call decodes all T steps, as in bench.py).
Each call is timed with CUDA events around the whole library call (encoder + decode + finalize).

    python profiles/nbest_bench.py [--calls 30] [--out profiles/nbest_bench.json]
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


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--beam", type=int, default=5)
    ap.add_argument("--max-len", type=int, default=150)
    ap.add_argument("--calls", type=int, default=30, help="timed calls of each form")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    cfg = ModelConfig()
    m = FormulaRecognitionModel(cfg.vocab_size)
    m.load_state_dict(synth_state_dict(cfg, seed=0, eos_bias_sigma=0.0))
    imgs = synth_images(8, seed=1234).cuda().repeat((a.batch + 7) // 8, 1, 1, 1)[: a.batch].contiguous()
    forms = {
        "generate": lambda: m.generate(imgs, max_len=a.max_len, beam_size=a.beam),
        "generate_nbest": lambda: m.generate_nbest(imgs, beam_size=a.beam, n_best=a.beam, max_len=a.max_len),
    }
    for f in forms.values():                      # warm-up: workspace, encoder graph capture, every shape
        for _ in range(3):
            f()
    torch.cuda.synchronize()
    ms = {k: [] for k in forms}
    for _ in range(a.calls):
        for k, f in forms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()                                   # ends in a host read of `steps`: the call has finished
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1))
    res = {"gpu": gpu_info(), "batch": a.batch, "beam": a.beam, "max_len": a.max_len, "calls": a.calls,
           "weights": "synthetic seed 0, eos never emitted"}
    for k, v in ms.items():
        res[k] = {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v),
                  "images_per_s": a.batch / statistics.median(v) * 1e3}
    res["nbest_over_best_only"] = res["generate_nbest"]["median_ms"] / res["generate"]["median_ms"]
    print(json.dumps(res, indent=1), flush=True)
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
