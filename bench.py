#!/usr/bin/env python
"""Benchmark of the image-to-LaTeX hot path, one BASELINE.json config per run (default: configs[1], the headline).

    python bench.py [--config 2|3|4|5] [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

  --config 2  Swin-T + 8-layer decoder, greedy, 256 images per GPU, T = 150              (BASELINE.json configs[1])
  --config 3  the same model, beam search (beam 5), 64 images per GPU, T = 150             (configs[2])
  --config 4  ResNet-18 + TransformerEncoder variant, greedy, 256 images per GPU, T = 150   (configs[3]; the encoder
              attends ACROSS the batch, so N GPUs = N replicas each with its own 256-image batch)
  --config 5  one point of the sweep: greedy, 1024 images per GPU, max LaTeX length 256      (configs[4])

One "step" = one pass of the hot path over one batch of synthetic rasterised stroke images per GPU: encoder ->
KV-cached decode (argmax / beam top-k on the device) -> token ids (N > 1: + the NCCL all-gather of the ids, the path's
only collective).  Prints ONE JSON line (rank 0).

  value        images/s, whole job, images already resident in HBM when the timed region starts (CUDA events, max over
               ranks, L2 flushed between steps)
  e2e          images/s through the public API with HOST buffers: every step copies its pinned uint8 images to the
               device (on a copy stream, overlapping the previous step's decode: two device buffers), preprocesses,
               encodes, decodes and copies its ids back to pinned host memory; L2 flushed between steps as for `value`
  roofline     the decode kernel against the measured HBM copy bandwidth on ALGORITHMIC bytes (SURVEY.md 8d /
               DESIGN.md); `encoder` sub-object: tensor roofline of the encoder
  cpu_baseline the oracle port of the reference greedy loop (src/inference.py) on the host cores (N = 1 only), plus
               the B = 1 latency of src/predict.py:49-67 (BASELINE.json configs[0]) beside `p50_ms_per_image_b1`

`--impl reference` times only that CPU path on the same config (the reference is pure Python over torch/torchvision
and does not exist on the GPU box; its algorithm is restated in oracle/ and pinned against the real reference by
oracle/make_golden.py).

`--dump-outputs DIR` writes what the timed path returned in its last timed step as float32 .npy files, so that two
builds can be compared output for output (inputs and weights are seeded, identical from run to run):
  tokens       [images, 1+T] token ids (column 0 = sos, pad past the step count; N > 1: all ranks' images)
  steps        decode steps executed (N > 1: one per rank)
  score        beam search only: the best hypothesis' score of each of rank 0's images
  tokens_rows  only when tokens alone would pass 64 MB: the fixed, seeded sample of rows kept in tokens
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

CONFIGS = {
    2: dict(arch="swin", batch=256, T=150, beam=1, baseline_index=1,
            workload="swin_t+8L-decoder greedy decode, B=256/GPU, T=150, V=5075, d_model=256 (BASELINE.json configs[1])"),
    3: dict(arch="swin", batch=64, T=150, beam=5, baseline_index=2,
            workload="swin_t+8L-decoder beam search (beam=5), B=64/GPU, T=150, V=5075 (BASELINE.json configs[2])"),
    4: dict(arch="res18", batch=256, T=150, beam=1, baseline_index=3,
            workload="resnet18+transformer-encoder variant (src/model_res18trans.py) greedy, B=256/GPU, T=150 "
                     "(BASELINE.json configs[3]); replicas with local batches"),
    5: dict(arch="swin", batch=1024, T=256, beam=1, baseline_index=4,
            workload="swin_t+8L-decoder greedy, sweep point B=1024/GPU x max LaTeX length 256 (BASELINE.json configs[4]; "
                     "config.max_seq_len raised to 256 before the model is built, SURVEY.md D6)"),
}
# bounded CPU samples (images per repetition) of the reference arm / cpu_baseline leg, per config
CPU_SAMPLE = {2: 8, 3: 2, 4: 8, 5: 2}
ENC_GFLOP = {"swin": 6.515, "res18": 2.24}       # reference-executed per image (SURVEY.md 8d; res18: 2.13 trunk + 0.11 encoder layers)
ENC_GFLOP_MINIMAL = {"swin": 5.498, "res18": 2.24}
MEM_TOKENS = {"swin": 30, "res18": 10}
DEC_WEIGHT_PARAMS = 7_630_547
DUMP_LIMIT_BYTES = 64 << 20


def peaks():
    p = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}
    f = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(f):
        try:
            d = json.load(open(f))
            p.update({k: d[k] for k in ("hbm_gbs", "bf16_tflops", "bf16_tflops_sustained") if k in d})
            p["source"] = "measured"
        except Exception:
            pass
    return p


def decode_algorithmic_bytes(images: int, T: int, beam: int = 1, S: int = 30, layers=8, d=256,
                             weight_params=DEC_WEIGHT_PARAMS) -> float:
    """SURVEY.md 8d, 2-byte KV: per step the cross K+V of an IMAGE is read once (L*S*2*d*2 B, shared by its beam
    hypotheses); every hypothesis reads L*2*d*2 B per cached position and appends L*2*d*2 B; the decoder weights
    (2 bytes per parameter) are read once per step per device.  The beam's parent reorder is implementation
    overhead, not counted."""
    cross = layers * S * 2 * d * 2
    per_pos = layers * 2 * d * 2
    hyp = sum(per_pos * t + per_pos for t in range(1, T + 1))
    return images * cross * T + images * beam * hyp + weight_params * 2 * T


def kernel_source_sha():
    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "handwritten_math_ocr_api_b200", "csrc")
    for f in ("decode_persistent.cu", "decode_persistent.cuh"):
        with open(os.path.join(csrc, f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def decode_traffic_from_ncu(batch: int, T: int, beam: int):
    """(dram__bytes_read.sum + dram__bytes_write.sum of the decode-kernel launches of ONE step, where it comes from).
    The number is NOT measured by this run (ncu replays kernels and cannot sit inside a timed run): it is read from the
    committed capture profiles/decode_traffic.json, and only while the decode kernel's sources are the ones that
    capture was taken with (sha256 recorded by profiles/summarize_ncu.py); otherwise null."""
    f = os.path.join(ROOT, "profiles", "decode_traffic.json")
    try:
        d = json.load(open(f))
    except Exception:
        return None, "no capture (profiles/decode_traffic.json missing)"
    if d.get("batch") != batch or d.get("max_len") != T or beam != 1:
        return None, "no capture for this workload (profiles/decode_traffic.json is B=%s, T=%s, greedy)" % (d.get("batch"), d.get("max_len"))
    sha = d.get("kernel_source_sha256")
    if sha is None or sha != kernel_source_sha():
        return None, "stale: profiles/decode_traffic.json (%s) was captured with other decode-kernel sources" % d.get("source")
    return d["dram_bytes_per_step"], "profiles/decode_traffic.json (%s, ncu capture of this kernel source, sha256 %s)" % (d.get("source"), sha[:12])


def dump_outputs(out_dir: str, tokens, steps, score=None):
    """Write the outputs of one step as DIR/<name>.npy (float32: token ids and step counts are exact), at most
    DUMP_LIMIT_BYTES in all; past that, `tokens` keeps a fixed, seeded sample of its rows, listed in tokens_rows.npy."""
    import numpy as np
    arrays = {"steps": steps.cpu().numpy().astype(np.float32)}
    if score is not None:
        arrays["score"] = score.cpu().numpy().astype(np.float32)
    tok = tokens.cpu().numpy().astype(np.float32)
    budget = DUMP_LIMIT_BYTES - sum(a.nbytes for a in arrays.values()) - 4 * 4096       # 4096: room for .npy headers
    if tok.nbytes > budget:
        keep = budget // (tok[0].nbytes + 4)
        rows = np.sort(np.random.default_rng(0).choice(tok.shape[0], keep, replace=False))
        arrays["tokens_rows"] = rows.astype(np.float32)
        tok = tok[rows]
    arrays["tokens"] = tok
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# CPU baseline (oracle port of the reference loops) - the ONLY place bench.py executes oracle/
# --------------------------------------------------------------------------------------------------
def cpu_reference_sample(config: int, reps: int, warmup: int):
    """One repetition = the reference's batched greedy loop (src/inference.py:7-25: encoder once, full-prefix decoder
    call per step) on CPU_SAMPLE[config] images of the config's workload; config 3 (beam search does not exist in
    the reference) runs the oracle's beam-search definition (KV-cached) instead."""
    from oracle import decode as odec
    from oracle.arch import ModelConfig
    from oracle.synth import synth_images
    c = CONFIGS[config]
    n_images, max_len = CPU_SAMPLE[config], c["T"]
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = ModelConfig(max_seq_len=max(150, max_len))
    imgs = synth_images(n_images, seed=1234)
    if c["arch"] == "res18":
        from handwritten_math_ocr_api_b200.synthetic import synth_pos_table, synth_state_dict_res18
        from oracle import res18_model as R18
        sd = synth_state_dict_res18(cfg, seed=0, eos_bias_sigma=0.0)
        dsd = R18._as_swin_decoder_sd(sd)
        pos = synth_pos_table(cfg.d_model, seed=0)

        def run():
            enc = R18.encoder_forward(imgs, sd, cfg, pos)
            return odec.greedy_batched(None, dsd, cfg, max_len=max_len, enc_out=enc)
        what = "oracle port of src/inference.py over src/model_res18trans.py (full-prefix recompute, torch eager fp32)"
    else:
        from oracle.synth import synth_state_dict
        sd = synth_state_dict(cfg, seed=0, eos_bias_sigma=0.0)
        if c["beam"] > 1:
            from oracle.ref_model import encoder_forward

            def run():
                return odec.beam_search(encoder_forward(imgs, sd), sd, cfg, beam=c["beam"], max_len=max_len)[0]
            what = ("oracle beam search (beam %d, KV-cached; the reference has no beam search, SURVEY.md D2), "
                    "torch eager fp32" % c["beam"])
        else:
            def run():
                return odec.greedy_batched(imgs, sd, cfg, max_len=max_len)     # src/inference.py:7-25 restated
            what = "oracle port of src/inference.py (full-prefix recompute, torch eager fp32)"
    times = []
    with torch.no_grad():
        for i in range(warmup + reps):
            t0 = time.perf_counter()
            ys = run()
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    steps = ys.shape[1] - 1
    return {"times": times, "images": n_images, "tokens": n_images * steps, "cores": torch.get_num_threads(),
            "sample": f"{n_images} images x {max_len} steps in one batch per repetition, {what}", "ys": ys}


def cpu_b1_latency(reps: int = 2):
    """BASELINE.json configs[0]: ONE image through src/predict.py:49-67 (B = 1, full-prefix recompute, 150 steps) on
    the host cores - the CPU number beside `p50_ms_per_image_b1`."""
    from oracle import decode as odec
    from oracle.arch import ModelConfig
    from oracle.synth import synth_images, synth_state_dict
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = ModelConfig()
    sd = synth_state_dict(cfg, seed=0, eos_bias_sigma=0.0)
    img = synth_images(1, seed=1234)
    ts = []
    with torch.no_grad():
        for _ in range(reps):
            t0 = time.perf_counter()
            odec.greedy_single(img, sd, cfg, max_len=150)
            ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


def run_reference(args, rank):
    if rank != 0:
        return
    c = CONFIGS[args.config]
    r = cpu_reference_sample(args.config, reps=args.steps, warmup=min(args.warmup, 1))
    mean = sum(r["times"]) / len(r["times"])
    ips = r["images"] / mean
    line = {
        "impl": "reference", "metric": "images_per_sec", "value": ips, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": mean * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "tokens_per_sec": r["tokens"] / mean,
        "config": {"workload": c["workload"] + " - CPU sample", "batch_per_step": r["images"], "max_len": c["T"],
                   "beam": c["beam"], "bench_config": args.config},
        "cpu_baseline": {"value": ips, "unit": "images/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
        "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.dump_outputs:
        ys = r["ys"]
        dump_outputs(args.dump_outputs, ys, torch.tensor([ys.shape[1] - 1]))
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def build_model(c, dev):
    from handwritten_math_ocr_api_b200.config import Config
    from handwritten_math_ocr_api_b200.layout import ModelConfig
    T = c["T"]

    class BenchConfig(Config):
        max_seq_len = max(150, T)

    cfg = ModelConfig(max_seq_len=max(150, T))
    if c["arch"] == "res18":
        from handwritten_math_ocr_api_b200.model_res18trans import FormulaRecognitionModel
        from handwritten_math_ocr_api_b200.synthetic import synth_pos_table, synth_state_dict_res18
        model = FormulaRecognitionModel(cfg.vocab_size, config=BenchConfig(), device=dev)
        model.load_state_dict(synth_state_dict_res18(cfg, seed=0, eos_bias_sigma=0.0))
        model.set_pos_table(synth_pos_table(cfg.d_model, seed=0))       # the reference re-draws it per call (D7): pinned here
    else:
        from handwritten_math_ocr_api_b200 import FormulaRecognitionModel
        from handwritten_math_ocr_api_b200.synthetic import synth_state_dict
        model = FormulaRecognitionModel(cfg.vocab_size, config=BenchConfig(), device=dev)
        model.load_state_dict(synth_state_dict(cfg, seed=0, eos_bias_sigma=0.0))   # never emits eos: exactly B*T tokens
    return model, cfg


def run_ours(args, rank, local_rank, world):
    import torch.distributed as dist
    from handwritten_math_ocr_api_b200 import _lib
    from handwritten_math_ocr_api_b200.parallel import gather_tokens_device
    from handwritten_math_ocr_api_b200.preprocess import preprocess_u8
    from handwritten_math_ocr_api_b200.synthetic import synth_images, synth_images_u8

    c = dict(CONFIGS[args.config])
    if args.batch:
        c["batch"] = args.batch
    if args.max_len:
        c["T"] = args.max_len
    B, T, beam, arch = c["batch"], c["T"], c["beam"], c["arch"]
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    model, cfg = build_model(c, dev)
    host_u8 = synth_images_u8(B, seed=1234 + rank).pin_memory()      # the rendered strokes as they come: uint8 96x320
    dev_imgs = synth_images(B, seed=1234 + rank).to(dev)             # = ToTensor + Normalize(0.5, 0.5) of host_u8
    lib = _lib.load()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)    # > 126 MB L2

    def decode(x):
        out = model.generate_device(x, max_len=T, beam_size=beam)
        return out[0], out[1]

    last = {}      # device outputs of the latest step_device() call, for --dump-outputs

    def step_device():
        out = model.generate_device(dev_imgs, max_len=T, beam_size=beam)
        tok, st = out[0], out[1]
        if world > 1:      # stream-ordered: decode -> the path's only collective (NCCL all-gather of the ids)
            tok, st = gather_tokens_device(tok, st)
        last.update(tokens=tok, steps=st, score=out[3] if beam > 1 else None)
        return tok, int(st.max().item())       # one host read per step

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = lib.hmocr_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    enc_ms, dec_ms = [], []
    barrier()
    wall0 = time.perf_counter()
    for i in range(args.steps):
        flush.fill_(i & 0xFF)                         # evict L2 between timed iterations (not timed)
        ev[i][0].record()
        tokens, steps = step_device()
        ev[i][1].record()
        e_ms, d_ms = model.last_timings_ms()          # CUDA events recorded by the library on this stream
        enc_ms.append(e_ms); dec_ms.append(d_ms)
    barrier()
    wall = time.perf_counter() - wall0
    timed_outputs = dict(last)
    launches = lib.hmocr_launch_count() - launches0
    clocks = sampler.stop()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    t = torch.tensor([sum(step_ms) / len(step_ms), sum(enc_ms) / len(enc_ms), sum(dec_ms) / len(dec_ms)],
                     dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step, ms_enc, ms_dec = t.tolist()
    assert steps == T, f"workload must run exactly {T} steps, ran {steps}"

    # ---- end to end through the public API with host buffers -------------------------------------
    # Every step: pinned uint8 images -> device (copy stream; two device buffers, so the copy of step i+1 runs under
    # the decode of step i) -> ToTensor/Normalize on the device -> encoder -> decode -> (N > 1: all-gather of the ids)
    # -> THIS rank's ids -> pinned host memory.  L2 is flushed between steps exactly as for `value`.
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream()
    u8_dev = [torch.empty_like(host_u8, device=dev) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    tok_host = [torch.empty(B, T + 1, dtype=torch.int64).pin_memory() for _ in range(2)]
    steps_host = [torch.zeros(1, dtype=torch.int32).pin_memory() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]

    def upload(i):
        s = i & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[s])                   # the buffer's previous reader has finished
            u8_dev[s].copy_(host_u8, non_blocking=True)
            ready[s].record(copy_stream)

    def e2e_loop(n):
        for s in range(2):
            consumed[s].record(main_stream)
        upload(0)
        for i in range(n):
            s = i & 1
            if i + 1 < n:
                upload(i + 1)
            flush.fill_(i & 0xFF)
            main_stream.wait_event(ready[s])
            x = preprocess_u8(model, u8_dev[s])
            consumed[s].record(main_stream)
            tok, st = decode(x)
            if world > 1:
                all_tok, st = gather_tokens_device(tok, st)       # the collective stays in the timed region
            if i >= 2:
                done[s].synchronize()                             # the host consumes step i-2's ids before its buffer is reused
            tok_host[s].copy_(tok, non_blocking=True)             # each rank hands ITS shard to its host
            steps_host[s].copy_(st.max().to(torch.int32).reshape(1), non_blocking=True)
            done[s].record(main_stream)
        main_stream.synchronize()

    e2e_loop(2)
    barrier()
    e0 = time.perf_counter()
    e2e_loop(args.steps)
    barrier()
    e2e_s = (time.perf_counter() - e0) / args.steps
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = te.item()
    assert int(steps_host[(args.steps - 1) & 1][0]) == T

    # serial form through the C ABI's host-buffer entry point (H2D, generate, D2H, sync per call), N = 1, Swin greedy/beam
    e2e_cabi = None
    if world == 1 and arch == "swin":
        import ctypes as C
        th, sh = tok_host[0], steps_host[0]

        def step_cabi():
            _lib.check(lib.hmocr_generate_host_u8(model._handle(), C.c_void_p(host_u8.data_ptr()), B, T, beam,
                                                  C.c_void_p(th.data_ptr()), None, C.c_void_p(sh.data_ptr()),
                                                  None, C.c_void_p(torch.cuda.current_stream().cuda_stream)),
                       "generate_host_u8")
        step_cabi()
        torch.cuda.synchronize()
        c0 = time.perf_counter()
        for i in range(args.steps):
            flush.fill_(i & 0xFF)
            step_cabi()
        torch.cuda.synchronize()
        e2e_cabi = B / ((time.perf_counter() - c0) / args.steps)

    # ---- B=1 latency (p50 per-image latency of BASELINE.json's metric) -----------------------------
    lat = []
    one = dev_imgs[:1].contiguous()
    for i in range(2 + 5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        model.generate(one, max_len=T, beam_size=beam)
        torch.cuda.synchronize()
        if i >= 2:
            lat.append((time.perf_counter() - t0) * 1e3)

    if rank == 0:
        pk = peaks()
        total_imgs = B * world
        value = total_imgs / (ms_step * 1e-3)
        dec_bytes = decode_algorithmic_bytes(B, T, beam, MEM_TOKENS[arch])
        ach = dec_bytes / (ms_dec * 1e-3) / 1e9
        enc_tf = ENC_GFLOP[arch] * 1e9 * B / (ms_enc * 1e-3) / 1e12
        traffic, traffic_source = decode_traffic_from_ncu(B, T, beam)
        # launches of the persistent kernel per step: one when every cluster of the batch is co-resident (the kernel
        # stops by itself), 16-step launches for multi-wave batches (engine.cu generate_persistent)
        import ctypes as _C
        _mc = _C.c_int()
        lib.hmocr_decode_max_clusters(_C.byref(_mc))
        _rpc = 8 if beam == 1 else beam * (8 // beam)
        n_launch = 1 if -(-(B * beam) // _rpc) <= _mc.value else -(-T // 16)
        line = {
            "metric": "images_per_sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
            "tokens_per_sec": total_imgs * T / (ms_step * 1e-3),
            "p50_ms_per_image_b1": statistics.median(lat), "ms_per_image_at_batch": ms_step / B,
            "encoder_ms": ms_enc, "decode_ms": ms_dec, "decode_us_per_step": ms_dec * 1e3 / T,
            "wall_ms_per_step": wall * 1e3 / args.steps,
            "config": {"workload": c["workload"], "bench_config": args.config, "batch_per_gpu": B, "max_len": T,
                       "beam": beam, "l2_flush_between_steps": True,
                       "weights": "synthetic seed 0 (handwritten_math_ocr_api_b200/synthetic.py, eos never emitted)",
                       "parallelism": f"dp{world}" if arch == "swin" else f"{world} replicas with local batches"},
            "roofline": {"bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                         "frac": ach / pk["hbm_gbs"], "traffic": traffic, "traffic_source": traffic_source,
                         "peak_source": pk["source"],
                         "kernel": "decode_persistent_kernel: the decode phase of one step = %d launch(es) of the persistent "
                                   "cluster kernel (+ memory K/V projection); bytes and CUDA-event time are summed over "
                                   "them; 2-byte (fp16) KV caches" % n_launch,
                         "algorithmic_bytes_per_step": dec_bytes,
                         "encoder": {"bound": "tensor", "achieved": enc_tf, "peak": pk["bf16_tflops_sustained"],
                                     "unit": "TFLOP/s", "frac": enc_tf / pk["bf16_tflops_sustained"],
                                     "gflop_per_image": ENC_GFLOP[arch],
                                     "gflop_per_image_minimal": ENC_GFLOP_MINIMAL[arch]}},
            "e2e": {"value": total_imgs / e2e_s, "unit": "images/s", "h2d_bytes_per_step": B * 96 * 320,
                    "d2h_bytes_per_step": B * (T + 1) * 8 + 4,
                    "input": "pinned uint8 [B,96,320] rendered strokes, copied on a copy stream into one of two device "
                             "buffers (overlaps the previous step's decode); ToTensor + Normalize(0.5,0.5), encoder and "
                             "decode on the device; each rank's ids back to its pinned host buffer; L2 flushed between steps",
                    "serial_c_abi_images_per_sec": e2e_cabi},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if beam > 1:
            line["emitted_tokens_per_sec"] = line["tokens_per_sec"]
            line["hypothesis_tokens_per_sec"] = line["tokens_per_sec"] * beam
        if world == 1 and not args.no_cpu:
            r = cpu_reference_sample(args.config, reps=2 if args.config in (3, 5) else 3, warmup=0)
            m = sum(r["times"]) / len(r["times"])
            line["cpu_baseline"] = {"value": r["images"] / m, "unit": "images/s", "cores": r["cores"], "kind": "port",
                                    "sample": r["sample"] + f", mean of {len(r['times'])} repetitions"}
            if args.config == 2:
                line["cpu_baseline"]["b1_p50_ms"] = cpu_b1_latency()
                line["cpu_baseline"]["b1_sample"] = ("one image, 150 greedy steps, oracle port of src/predict.py:49-67 "
                                                     "(BASELINE.json configs[0]), median of 2")
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, **timed_outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json config (2 = headline)")
    ap.add_argument("--batch", type=int, default=0, help="override the config's images per GPU")
    ap.add_argument("--max-len", type=int, default=0, help="override the config's decode length")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus:
        if args.gpus > 1 and world == 1:
            # launched without torchrun: re-exec under it
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                   "--master-addr", "127.0.0.1", "--master-port", "29541", os.path.abspath(__file__)] + sys.argv[1:]
            sys.exit(subprocess.call(cmd))
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
