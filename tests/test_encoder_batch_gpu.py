"""GPU: both encoders at the batch sizes the benchmark runs, on the benchmark's own checkpoint and images.

bench.py runs the Swin encoder at 256 images (configs 2 and 3 at 256 and 64) and 1024 (config 5), the ResNet-18
variant at 256 (config 4).  At those batches the engine takes paths that a 2-4 image test never reaches:
  * window attention: the grid is capped at 296 / heads CTAs per head, so from B = 17 (stage 1), 33 (stage 2),
    49 (stage 4) and 65 (stage 3) a warp loops over more than one window, reusing its gather tiles;
  * the CTA-pair GEMM (K >= 1024, N % 192 == 0, M >= 512): stage-3 fc2 from B = 5, stage-4 fc2 and the last
    patch-merge reduction from B = 18;
  * the stage-1 GEMMs and the fused MLP at up to two million rows (tens of tiles per CTA);
  * ResNet-18: attention across the batch with T = B = 256 keys (four 64-key chunks), 64 four-image conv tiles in
    layer 4, and the 256-image limit;
  * the C ABI's host-buffer entry points (bench.py's serial_c_abi_images_per_sec).

What is promised decides what is checked: a Swin image's features do not depend on its batch-mates (SURVEY.md 8e),
so they are compared BIT FOR BIT across batches; against the float64 oracle (where only a tolerance is promised) the
bounds are those of test_model_gpu.py / test_res18_gpu.py, with what was measured here recorded beside them.
"""
import ctypes as C

import pytest
import torch

from gpu_utils import P, S

pytestmark = pytest.mark.gpu

FEAT_TOL = 1e-2            # Swin features, test_model_gpu.py
RES18_FEAT_TOL = 1.5e-2    # ResNet-18 variant features, test_res18_gpu.py
RES18_FEAT_TOL_MAX_256 = 1e-1   # its worst image at 256 (test_res18_features_at_the_serving_batch_against_float64)
SWIN_BATCHES = [17, 49, 65, 256, 1024, 1025]
MAX_LEN = 24


def _check(rc, what):
    from handwritten_math_ocr_api_b200 import _lib
    _lib.check(rc, what)


@pytest.fixture(scope="module")
def bench_sd(cfg):
    """bench.py's Swin checkpoint (never emits eos: every decode runs max_len steps)."""
    from handwritten_math_ocr_api_b200.synthetic import synth_state_dict
    return synth_state_dict(cfg, seed=0, eos_bias_sigma=0.0)


def _swin_engine(sd, cfg):
    from handwritten_math_ocr_api_b200 import FormulaRecognitionModel
    m = FormulaRecognitionModel(cfg.vocab_size)
    m.load_state_dict(sd)
    return m.eval()


@pytest.fixture(scope="module")
def swin(bench_sd, cfg):
    return _swin_engine(bench_sd, cfg)


@pytest.fixture(scope="module")
def images():
    """bench.py's images: image i depends only on (seed, i), so images[:B] is synth_images(B, 1234)."""
    from handwritten_math_ocr_api_b200.synthetic import synth_images
    return synth_images(max(SWIN_BATCHES), seed=1234)


def _f64(sd):
    return {k: (v.to("cuda", torch.float64) if v.is_floating_point() else v.cuda()) for k, v in sd.items()}


# ---- the Swin schedule rebuilt from the exported kernels --------------------------------------------------------
def swin_stages(imgs, dsd):
    """engine.cu encode_impl at any batch, one exported kernel at a time (patch embed, LayerNorm, qkv / proj / MLP /
    reduction GEMMs, window attention, fused MLP of stages 1-2, patch-merge LayerNorm), on the fp16 weights the engine
    uploads.  Returns the residual stream after patch embed and after every block and merge ([B, H, W, C] f32, the
    layout of oracle.ref_model.encoder_stages) and the projected features [B, 30, 256]: the same kernels on the same
    operands in the same order, so the features are the bits of model.encoder."""
    from handwritten_math_ocr_api_b200 import _lib
    from oracle.arch import DEPTHS, HEADS
    lib = _lib.load()
    fp = "encoder.features."
    B = imgs.shape[0]
    H, W, C_ = 24, 80, 96

    def half(k):
        return dsd[k].half().contiguous()

    def gemm(a16, w16, bias=None, act=0, x=None, out16=False):
        """fp16 [M, K] x [N, K]^T: into x in place (x += ...) when given, else a new f32 or fp16 tensor."""
        M, K = a16.shape
        N = w16.shape[0]
        o16 = torch.empty(M, N, dtype=torch.float16, device="cuda") if out16 else None
        o32 = x if x is not None else (None if out16 else torch.empty(M, N, device="cuda"))
        _check(lib.hmocr_gemm_f16(P(a16), K, M, K, P(w16), N, P(bias), act, P(x), N if x is not None else 0, P(o32), N,
                                  P(o16), N, None, None, 0, S()), "hmocr_gemm_f16")
        return o16 if out16 else o32

    def layernorm(x, prefix):
        xn = torch.empty(x.shape, dtype=torch.float16, device="cuda")
        _check(lib.hmocr_layernorm(P(x), x.shape[0], x.shape[1], P(dsd[prefix + ".weight"]), P(dsd[prefix + ".bias"]),
                                   P(xn), None, S()), "hmocr_layernorm")
        return xn

    x = torch.empty(B * H * W, C_, device="cuda")
    _check(lib.hmocr_patch_embed(P(imgs), B, P(dsd[fp + "0.0.weight"].reshape(96, 16).contiguous()), P(dsd[fp + "0.0.bias"]),
                                 P(dsd[fp + "0.2.weight"]), P(dsd[fp + "0.2.bias"]), P(x), S()), "hmocr_patch_embed")
    stages = [x.reshape(B, H, W, C_).clone()]
    for s in range(4):
        fi, heads = 1 + 2 * s, HEADS[s]
        for j in range(DEPTHS[s]):
            bp = f"{fp}{fi}.{j}."
            qkv = gemm(layernorm(x, bp + "norm1"), half(bp + "attn.qkv.weight"), dsd[bp + "attn.qkv.bias"], out16=True)
            idx = dsd[bp + "attn.relative_position_index"]
            rel = dsd[bp + "attn.relative_position_bias_table"][idx].reshape(49, 49, heads).permute(2, 0, 1).contiguous()
            ctx = torch.empty(x.shape, dtype=torch.float16, device="cuda")
            _check(lib.hmocr_window_attention(P(qkv), P(dsd[bp + "attn.qkv.bias"]), P(rel), B, H, W, C_, heads,
                                              3 if j % 2 else 0, P(ctx), S()), "hmocr_window_attention")
            gemm(ctx, half(bp + "attn.proj.weight"), dsd[bp + "attn.proj.bias"], x=x)
            xn = layernorm(x, bp + "norm2")
            if C_ in (96, 192):            # engine.cu: mlp_fused (default) where swin_mlp_supported(C)
                w1, w2 = half(bp + "mlp.0.weight"), half(bp + "mlp.3.weight")      # alive until the launch
                _check(lib.hmocr_swin_mlp(P(xn), x.shape[0], C_, P(w1), P(dsd[bp + "mlp.0.bias"]), P(w2),
                                          P(dsd[bp + "mlp.3.bias"]), P(x), S()), "hmocr_swin_mlp")
            else:
                hid = gemm(xn, half(bp + "mlp.0.weight"), dsd[bp + "mlp.0.bias"], act=1, out16=True)
                gemm(hid, half(bp + "mlp.3.weight"), dsd[bp + "mlp.3.bias"], x=x)
            stages.append(x.reshape(B, H, W, C_).clone())
        if s < 3:
            mp = f"{fp}{fi + 1}."
            xn = torch.empty(x.shape[0] // 4, 4 * C_, dtype=torch.float16, device="cuda")
            _check(lib.hmocr_patch_merge_ln(P(x), B, H, W, C_, P(dsd[mp + "norm.weight"]), P(dsd[mp + "norm.bias"]), P(xn),
                                            S()), "hmocr_patch_merge_ln")
            x = gemm(xn, half(mp + "reduction.weight"))
            H, W, C_ = H // 2, W // 2, 2 * C_
            stages.append(x.reshape(B, H, W, C_).clone())
    feats = gemm(x.half(), half("encoder.projection.weight"), dsd["encoder.projection.bias"])
    torch.cuda.synchronize()
    return stages, feats.reshape(B, H * W, -1)


# Bound of each stage's residual stream against the oracle, relative to max(1, the stage's largest magnitude): patch
# embed is an fp32 path (1e-4, as before); every later stage carries the fp16 rounding (2^-11 relative) of the GEMM and
# attention operands of the blocks before it, bounded like an fp32 GEMM output of test_kernels_gpu.py::test_gemm_plain
# (2e-3 relative).  Measured on a B200 (1000 W): at most 8.6e-4 at B = 65 and at B = 2 (the golden images).
STAGE_REL_TOL = [1e-4] + [2e-3] * 15


def stage_errors(got, want):
    """Per-stage max-abs error relative to max(1, max |want|)."""
    return [float((g.double() - w.double()).abs().max()) / max(1.0, float(w.abs().max())) for g, w in zip(got, want)]


def assert_stages_close(got, want):
    errs = stage_errors(got, want)
    print("per-stage error relative to the stage's magnitude:", " ".join(f"{e:.2e}" for e in errs))
    bad = [(i, e, t) for i, (e, t) in enumerate(zip(errs, STAGE_REL_TOL)) if not e < t]
    assert not bad, f"first stage out of bounds (index in oracle.ref_model.encoder_stages, error, bound): {bad[0]}"


def _oracle_in_chunks(fn, imgs, chunk=32):
    with torch.no_grad():
        return [fn(imgs[i:i + chunk].double()) for i in range(0, imgs.shape[0], chunk)]


# ---- per-image bits at every batch regime ---------------------------------------------------------------------
@pytest.mark.parametrize("B", SWIN_BATCHES)
def test_swin_features_of_an_image_are_the_same_bits_at_every_batch(swin, images, B):
    """Rows {0, 1, B//2, B-1} and two seeded random rows of one B-image batch are the bits of the same image encoded
    alone and in a batch of four.  17 / 49 / 65 cross the window-loop start of stages 1 / 4 / 3 (65: all four stages
    loop), 256 and 1024 are the benchmark's batches (stage-1 GEMMs and fused MLP at 491,520 and 1,966,080 rows), 1025
    is one past the encoder-graph limit of generate()."""
    g = torch.Generator().manual_seed(B)
    rows = sorted({0, 1, B // 2, B - 1, *torch.randint(0, B, (2,), generator=g).tolist()})
    full = swin.encoder(images[:B].cuda())[rows]
    alone = torch.cat([swin.encoder(images[r:r + 1].cuda()) for r in rows])
    padded = rows + rows[:-len(rows) % 4]
    four = torch.cat([swin.encoder(images[padded[i:i + 4]].cuda()) for i in range(0, len(padded), 4)])
    for i, r in enumerate(rows):
        assert torch.equal(full[i], alone[i]), (r, float((full[i] - alone[i]).abs().max()))
        assert torch.equal(full[i], four[i]), (r, float((full[i] - four[i]).abs().max()))


# ---- features at 256 images against float64 -------------------------------------------------------------------
def test_swin_features_at_256_images_against_float64(swin, bench_sd, images):
    """The engine's [256, 30, 256] features against oracle.ref_model.encoder_forward in float64, per image.
    Measured on a B200 (1000 W), per-image max-abs error: max 4.4e-3, median 3.6e-3 (bound FEAT_TOL = 1e-2)."""
    from oracle import ref_model as R
    imgs = images[:256].cuda()
    feats = swin.encoder(imgs)
    dsd = _f64(bench_sd)
    ref = torch.cat(_oracle_in_chunks(lambda x: R.encoder_forward(x, dsd), imgs))
    per_image = (feats.double() - ref).abs().amax(dim=(1, 2))
    print(f"Swin features at B=256 vs float64: per-image max-abs error max {per_image.max():.3e}, "
          f"median {per_image.median():.3e}")
    assert (per_image < FEAT_TOL).all(), per_image.max().item()


# ---- the stage-level localiser --------------------------------------------------------------------------------
def test_swin_stages_at_65_images_against_float64(swin, bench_sd, images):
    """At B = 65 every stage's window attention loops over windows: every stage of the rebuilt schedule against the
    float64 oracle's, and the rebuilt schedule's features are the bits of model.encoder (so a failure of the batch
    tests above can be localised with swin_stages at the failing batch)."""
    from oracle import ref_model as R
    imgs = images[:65].cuda()
    dsd = {k: v.cuda() for k, v in bench_sd.items()}
    got, feats = swin_stages(imgs, dsd)
    assert torch.equal(feats, swin.encoder(imgs))
    d64 = _f64(bench_sd)
    chunks = _oracle_in_chunks(lambda x: R.encoder_stages(x, d64), imgs)
    want = [torch.cat(parts) for parts in zip(*chunks)]
    assert_stages_close(got, want)


# ---- the ResNet-18 variant at its serving batch ---------------------------------------------------------------
@pytest.fixture(scope="module")
def res18(cfg):
    from handwritten_math_ocr_api_b200.model_res18trans import FormulaRecognitionModel
    from handwritten_math_ocr_api_b200.synthetic import synth_pos_table, synth_state_dict_res18
    sd = synth_state_dict_res18(cfg, seed=0, eos_bias_sigma=0.0)
    m = FormulaRecognitionModel(cfg.vocab_size)
    m.load_state_dict(sd)
    return m.eval(), sd, synth_pos_table(256, seed=0)


@pytest.mark.parametrize("B", [256, 255])
def test_res18_features_at_the_serving_batch_against_float64(res18, cfg, images, B):
    """Attention across 256 (255) images, 64 four-image conv tiles in layer 4 (255: the last one ragged), against
    oracle.res18_model.encoder_forward in float64 with the same positional table.

    Measured on a B200 (1000 W), per-image max-abs error: B = 256 max 6.5e-2, median 1.1e-2; B = 255 max 6.5e-2,
    median 1.1e-2 (the same four images alone: at most 1.1e-2).  The typical image meets test_res18_gpu.py's
    FEAT_TOL = 1.5e-2; the worst does not, and that is the fp16 operands, not a kernel: the trunk's activations reach
    405 on this checkpoint (fp16 spacing 0.25 there), and float64 arithmetic with only the trunk's conv inputs,
    BN-folded weights and pooled output rounded to fp16 where the engine rounds them lands up to 1.0e-1 (median
    8.5e-3) from plain float64 at B = 256: 256-key attention across the batch amplifies a 2^-11 relative change of the
    trunk output that much.  So the median is held to FEAT_TOL and the worst image to that 1e-1."""
    from oracle import res18_model as R18
    m, sd, pos = res18
    imgs = images[:B].cuda()
    feats = m.encoder(imgs, pos)
    with torch.no_grad():
        ref = R18.encoder_forward(imgs.double(), _f64(sd), cfg, pos.to("cuda", torch.float64))
    per_image = (feats.double() - ref).abs().amax(dim=(1, 2))
    print(f"ResNet-18 features at B={B} vs float64: per-image max-abs error max {per_image.max():.3e}, "
          f"median {per_image.median():.3e}")
    assert per_image.median() < RES18_FEAT_TOL, per_image.median().item()
    assert (per_image < RES18_FEAT_TOL_MAX_256).all(), per_image.max().item()


def test_res18_generate_from_images_is_encoder_then_decode_at_256(res18, images):
    """generate(images) at B = 256 (call 1 eager, call 2 captures the encoder graph, call 3 replays it) returns the
    bits of generate(encoder_out=model.encoder(images))."""
    m, _, pos = res18
    imgs = images[:256].cuda()
    want = m.generate(encoder_out=m.encoder(imgs, pos), max_len=MAX_LEN, return_logprobs=True)
    for call in range(3):
        tok, steps, lp = m.generate(imgs, max_len=MAX_LEN, return_logprobs=True, pos_table=pos)
        assert steps == want[1] == MAX_LEN, call
        assert torch.equal(tok, want[0]) and torch.equal(lp, want[2]), call


def test_res18_refuses_257_images_and_keeps_working(res18, images):
    """The encoder attends across the batch, in one CTA per (position, head) that holds every key: more than 256 images
    are refused by name, and a refused call leaves the engine usable, at shapes it has not planned for yet too."""
    m, _, pos = res18
    four = images[:4].cuda()
    before = m.encoder(four, pos).clone()
    with pytest.raises(RuntimeError, match="batch 257 > 256 unsupported"):
        m.encoder(images[:257].cuda(), pos)
    with pytest.raises(RuntimeError, match="batch 257 > 256 unsupported"):
        m.generate(images[:257].cuda(), max_len=MAX_LEN, pos_table=pos)
    assert torch.equal(m.encoder(four, pos), before)
    tok, steps, lp = m.generate(four, max_len=2 * MAX_LEN, return_logprobs=True, pos_table=pos)
    want = m.generate(encoder_out=before, max_len=2 * MAX_LEN, return_logprobs=True)
    assert steps == want[1] and torch.equal(tok, want[0]) and torch.equal(lp, want[2])


# ---- the host-buffer entry points -----------------------------------------------------------------------------
@pytest.mark.parametrize("entry", ["hmocr_generate_host_u8", "hmocr_generate_host"])
def test_host_buffer_entry_points_at_256_images(swin, bench_sd, cfg, images, entry):
    """The C ABI's host-buffer forms (pinned images in, pinned tokens / steps / log-probs out) on a fresh engine,
    three calls (eager encoder, graph capture, graph replay): the results of preprocess_u8 + generate on the device."""
    from handwritten_math_ocr_api_b200 import _lib
    from handwritten_math_ocr_api_b200.preprocess import preprocess_u8
    from handwritten_math_ocr_api_b200.synthetic import synth_images_u8
    B = 256
    u8 = synth_images_u8(B, seed=1234).pin_memory()
    want_tok, want_steps, want_lp = swin.generate(preprocess_u8(swin, u8.cuda()), max_len=MAX_LEN, return_logprobs=True)
    src = u8 if entry.endswith("_u8") else images[:B].clone().pin_memory()
    m = _swin_engine(bench_sd, cfg)
    fn = getattr(_lib.load(), entry)
    for call in range(3):
        tok = torch.full((B, MAX_LEN + 1), -1, dtype=torch.int64).pin_memory()
        lp = torch.full((B, MAX_LEN), 1.0).pin_memory()
        steps = torch.full((1,), -1, dtype=torch.int32).pin_memory()
        _check(fn(m._handle(), C.c_void_p(src.data_ptr()), B, MAX_LEN, 1, C.c_void_p(tok.data_ptr()),
                  C.c_void_p(lp.data_ptr()), C.c_void_p(steps.data_ptr()), None, S()), entry)
        n = int(steps[0])
        assert n == want_steps, (call, n)
        assert torch.equal(tok[:, :n + 1], want_tok.cpu()) and torch.equal(lp[:, :n], want_lp.cpu()), call
