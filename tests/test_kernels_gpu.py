"""GPU: each hand-written kernel against plain torch fp32 / the oracle on identical tensors."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

from gpu_utils import P, S, gemm, gemm_ref  # noqa: E402


def _lib():
    from handwritten_math_ocr_api_b200 import _lib as L
    return L.load(), L


def _rand(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(*shape, device="cuda", generator=g) * scale)


# every (M, K, N) class on the hot path (SURVEY.md 2.2), shrunk in M to B=2 images, plus tails
GEMM_SHAPES = [
    (3840, 96, 288), (3840, 96, 96), (3840, 96, 384), (3840, 384, 96),          # stage 1
    (960, 384, 192), (960, 192, 576), (960, 192, 192), (960, 192, 768), (960, 768, 192),   # merge 1, stage 2
    (240, 768, 384), (240, 384, 1152), (240, 384, 384), (240, 384, 1536), (240, 1536, 384),  # merge 2, stage 3
    (60, 1536, 768), (60, 768, 2304), (60, 768, 768), (60, 768, 3072), (60, 3072, 768),   # merge 3, stage 4
    (60, 768, 256),                                                              # projection
    (256, 256, 768), (256, 256, 256), (256, 256, 512), (256, 512, 256), (256, 256, 5120),  # decoder step B=256
    (1, 256, 768), (7, 256, 5120), (129, 96, 96), (300, 256, 4096),             # ragged M
    (20000, 96, 288), (19000, 384, 96),                                          # many tiles per CTA (persistence)
    (491520, 96, 288),                                                           # stage-1 qkv at B=256
    (30720, 3072, 768),                                                          # stage-4 fc2 at B=1024 (CTA pair)
]


@pytest.mark.parametrize("M,K,N", GEMM_SHAPES)
def test_gemm_plain(M, K, N):
    a = _rand(M, K, seed=1).half()
    w = _rand(N, K, scale=K ** -0.5, seed=2).half()
    o32, o16 = gemm(a, w, out_f16=True)
    ref = gemm_ref(a, w)
    err = (o32 - ref).abs().max().item()
    assert err < 2e-3 * max(1.0, ref.abs().max().item()), err      # fp32 accumulation-order noise only
    assert (o16.float() - ref).abs().max().item() < 2e-2 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("bn", [64, 96, 128, 192, 256])
def test_gemm_every_tile_width(bn):
    M, K, N = 1000, 320, bn * 3
    a = _rand(M, K, seed=3).half()
    w = _rand(N, K, scale=K ** -0.5, seed=4).half()
    o32, _ = gemm(a, w, force_bn=bn)
    assert (o32 - gemm_ref(a, w)).abs().max().item() < 3e-3


@pytest.mark.parametrize("act", [0, 1, 2])
def test_gemm_bias_act_residual(act):
    M, K, N = 777, 384, 192
    a = _rand(M, K, seed=5).half()
    w = _rand(N, K, scale=K ** -0.5, seed=6).half()
    bias, res = _rand(N, seed=7), _rand(M, N, seed=8)
    o32, o16 = gemm(a, w, bias=bias, act=act, residual=res, out_f16=True)
    ref = gemm_ref(a, w, bias, act, res)
    assert (o32 - ref).abs().max().item() < 3e-3
    assert (o16.float() - ref).abs().max().item() < 5e-2


def test_gemm_residual_in_place():
    lib, L = _lib()
    M, K, N = 500, 96, 96
    a = _rand(M, K, seed=9).half()
    w = _rand(N, K, scale=K ** -0.5, seed=10).half()
    bias = _rand(N, seed=11)
    x = _rand(M, N, seed=12)
    ref = gemm_ref(a, w, bias, 0, x.clone())
    L.check(lib.hmocr_gemm_f16(P(a), K, M, K, P(w), N, P(bias), 0, P(x), N, P(x), N, None, 0, None, None, 0, S()), "gemm")
    torch.cuda.synchronize()
    assert (x - ref).abs().max().item() < 3e-3


@pytest.mark.parametrize("N,K", [(256, 256), (256, 512), (96, 96), (192, 768)])
def test_gemm_fused_layernorm(N, K):
    M = 300
    a = _rand(M, K, seed=13).half()
    w = _rand(N, K, scale=K ** -0.5, seed=14).half()
    bias, res = _rand(N, seed=15), _rand(M, N, seed=16)
    g, b = 1 + 0.2 * _rand(N, seed=17), 0.1 * _rand(N, seed=18)
    o32, o16 = gemm(a, w, bias=bias, residual=res, ln=(g, b), out_f16=True)
    ref = gemm_ref(a, w, bias, 0, res, (g, b))
    assert (o32 - ref).abs().max().item() < 3e-3
    assert (o16.float() - ref).abs().max().item() < 5e-2


@pytest.mark.parametrize("C_,M", [(96, 3840), (96, 128), (96, 1), (96, 130), (96, 40000), (192, 960), (192, 200), (192, 30000),
                                  (96, 491520), (192, 122880)])
def test_swin_mlp_fused(C_, M):
    """x <- x + fc2(GELU(fc1(xn))) in ONE kernel (hidden tile in TMEM / shared memory) against (a) plain torch fp32
    with the hidden activations rounded to fp16 where the kernel rounds them, (b) the two-GEMM path of the library
    (same arithmetic, same rounding points: equal up to fp32 summation order).  M covers one tile, a ragged last
    tile, a single row and many tiles per CTA (persistence, barrier phase wrap-around), up to stages 1 and 2 at B=256."""
    lib, L = _lib()
    xn = _rand(M, C_, seed=30).half()
    w1 = _rand(4 * C_, C_, scale=C_ ** -0.5, seed=31).half()
    w2 = _rand(C_, 4 * C_, scale=(4 * C_) ** -0.5, seed=32).half()
    b1, b2 = 0.3 * _rand(4 * C_, seed=33), 0.3 * _rand(C_, seed=34)
    x0 = _rand(M, C_, seed=35) * 2
    hid = torch.nn.functional.gelu(xn.float() @ w1.float().t() + b1).half()
    ref = x0 + hid.float() @ w2.float().t() + b2
    x = x0.clone()
    L.check(lib.hmocr_swin_mlp(P(xn), M, C_, P(w1), P(b1), P(w2), P(b2), P(x), S()), "swin_mlp")
    torch.cuda.synchronize()
    assert torch.isfinite(x).all()
    err = (x - ref).abs().max().item()
    assert err < 3e-3, err
    # the two-launch path: fc1 + GELU -> fp16 hidden in HBM, fc2 + residual in place
    _, h16 = gemm(xn, w1, bias=b1, act=1, out_f32=False, out_f16=True)
    x2 = x0.clone()
    L.check(lib.hmocr_gemm_f16(P(h16), 4 * C_, M, 4 * C_, P(w2), C_, P(b2), 0, P(x2), C_, P(x2), C_, None, 0, None, None,
                               0, S()), "gemm")
    torch.cuda.synchronize()
    assert (x - x2).abs().max().item() < 1e-3
    # a second call on the same buffers (tensor-map cache, barrier state of a fresh launch) gives the same result
    x3 = x0.clone()
    L.check(lib.hmocr_swin_mlp(P(xn), M, C_, P(w1), P(b1), P(w2), P(b2), P(x3), S()), "swin_mlp")
    torch.cuda.synchronize()
    assert torch.equal(x, x3)


def test_swin_mlp_rejects_other_widths():
    lib, L = _lib()
    xn = _rand(8, 384).half()
    w1, w2 = _rand(1536, 384).half(), _rand(384, 1536).half()
    b1, b2, x = _rand(1536), _rand(384), _rand(8, 384)
    rc = lib.hmocr_swin_mlp(P(xn), 8, 384, P(w1), P(b1), P(w2), P(b2), P(x), S())
    assert rc != 0 and b"unsupported" in lib.hmocr_last_error()


def test_gemm_rejects_bad_shapes():
    lib, L = _lib()
    a = _rand(8, 64).half()
    w = _rand(40, 64).half()
    out = torch.empty(8, 40, device="cuda")
    rc = lib.hmocr_gemm_f16(P(a), 64, 8, 64, P(w), 40, None, 0, None, 0, P(out), 40, None, 0, None, None, 0, S())
    assert rc != 0 and b"multiple of 32" in lib.hmocr_last_error()


@pytest.mark.parametrize("C_", [96, 192, 384, 768, 1536, 256])
def test_layernorm(C_):
    lib, L = _lib()
    rows = 1000
    x = _rand(rows, C_, seed=20) * 3 + 0.5
    g, b = 1 + 0.2 * _rand(C_, seed=21), 0.1 * _rand(C_, seed=22)
    o16 = torch.empty(rows, C_, dtype=torch.float16, device="cuda")
    o32 = torch.empty(rows, C_, dtype=torch.float32, device="cuda")
    L.check(lib.hmocr_layernorm(P(x), rows, C_, P(g), P(b), P(o16), P(o32), S()), "layernorm")
    torch.cuda.synchronize()
    ref = torch.nn.functional.layer_norm(x, (C_,), g, b, 1e-5)
    assert (o32 - ref).abs().max().item() < 2e-5
    assert (o16.float() - ref).abs().max().item() < 4e-2


def test_patch_embed_against_oracle(sd):
    from oracle import ref_model as R
    from oracle.synth import synth_images
    lib, L = _lib()
    imgs = synth_images(3).cuda()
    dsd = {k: v.cuda() for k, v in sd.items() if k.startswith("encoder.features.0.")}
    ref = R.patch_embed(imgs, dsd, "encoder.features.")
    x = torch.empty(3, 24, 80, 96, device="cuda")
    L.check(lib.hmocr_patch_embed(P(imgs), 3, P(dsd["encoder.features.0.0.weight"]), P(dsd["encoder.features.0.0.bias"]),
                                  P(dsd["encoder.features.0.2.weight"]), P(dsd["encoder.features.0.2.bias"]), P(x), S()),
            "patch_embed")
    torch.cuda.synchronize()
    assert (x - ref).abs().max().item() < 2e-5


@pytest.mark.parametrize("B,H,W,Cin", [(2, 24, 80, 96), (2, 12, 40, 192), (2, 6, 20, 384), (256, 24, 80, 96)])
def test_patch_merge_ln(B, H, W, Cin):
    lib, L = _lib()
    x = _rand(B, H, W, Cin, seed=30)
    g, b = 1 + 0.2 * _rand(4 * Cin, seed=31), 0.1 * _rand(4 * Cin, seed=32)
    out = torch.empty(B, H // 2, W // 2, 4 * Cin, dtype=torch.float16, device="cuda")
    L.check(lib.hmocr_patch_merge_ln(P(x), B, H, W, Cin, P(g), P(b), P(out), S()), "patch_merge_ln")
    torch.cuda.synchronize()
    cat = torch.cat([x[:, 0::2, 0::2], x[:, 1::2, 0::2], x[:, 0::2, 1::2], x[:, 1::2, 1::2]], -1)
    ref = torch.nn.functional.layer_norm(cat, (4 * Cin,), g, b, 1e-5)
    assert (out.float() - ref).abs().max().item() < 4e-2


@pytest.mark.parametrize("B", [2, 70])
@pytest.mark.parametrize("stage,shift", [(0, 0), (0, 3), (1, 0), (1, 3), (2, 0), (2, 3), (3, 0), (3, 3)])
def test_window_attention_against_oracle(stage, shift, B):
    """All four stage geometries incl. the suppressed H-shift (stage 3/4) and the 7x14 padded stage 4.  At B = 70 the
    grid's cap (296 / heads CTAs per head) makes every warp of every stage loop over more than one window."""
    from oracle import ref_model as R
    from oracle.arch import stage_dims
    lib, L = _lib()
    H, W, C_, heads = stage_dims()[stage]
    xn = _rand(B, H, W, C_, seed=40 + stage)
    bp = "b."
    dsd = {
        bp + "attn.qkv.weight": _rand(3 * C_, C_, scale=C_ ** -0.5, seed=50),
        bp + "attn.qkv.bias": 0.3 * _rand(3 * C_, seed=51),
        bp + "attn.relative_position_bias_table": _rand(169, heads, seed=52),
        bp + "attn.proj.weight": torch.eye(C_, device="cuda"),
        bp + "attn.proj.bias": torch.zeros(C_, device="cuda"),
    }
    from oracle.synth import relative_position_index
    idx = torch.from_numpy(relative_position_index()).cuda()
    dsd[bp + "attn.relative_position_index"] = idx
    # feed both sides the SAME fp16-rounded qkv so only the attention core is compared
    qkv = torch.nn.functional.linear(xn, dsd[bp + "attn.qkv.weight"], dsd[bp + "attn.qkv.bias"]).half()
    rel = dsd[bp + "attn.relative_position_bias_table"][idx].reshape(49, 49, heads).permute(2, 0, 1).contiguous()
    ctx = torch.zeros(B * H * W, C_, dtype=torch.float16, device="cuda")
    L.check(lib.hmocr_window_attention(P(qkv), P(dsd[bp + "attn.qkv.bias"]), P(rel), B, H, W, C_, heads, shift, P(ctx), S()),
            "window_attention")
    torch.cuda.synchronize()
    # oracle with a qkv Linear that reproduces the rounded qkv: run it on an identity-embedded input
    # instead: recompute from the rounded tensor by monkey-patching the linear through a hook
    ref = _oracle_attention_from_qkv(qkv.float().reshape(B, H, W, 3 * C_), dsd, bp, heads, shift)
    err = (ctx.float().reshape(B, H, W, C_) - ref).abs().max().item()
    assert err < 3e-2, err


def _oracle_attention_from_qkv(qkv, dsd, bp, heads, shift):
    """oracle.ref_model.window_attention with the qkv Linear factored out (padded rows = bias)."""
    from oracle import ref_model as R
    B, H, W, C3 = qkv.shape
    C_ = C3 // 3
    hd = C_ // heads
    Hp, Wp, sh, sw, src, valid, region = R.window_geometry(H, W, shift)
    nW, N = src.shape
    src, valid, region = src.cuda(), valid.cuda(), region.cuda()
    tok = qkv.reshape(B, H * W, C3)[:, src.reshape(-1), :]
    bias_row = dsd[bp + "attn.qkv.bias"].reshape(1, 1, C3)
    tok = torch.where(valid.reshape(1, -1, 1), tok, bias_row.expand_as(tok)).reshape(B * nW, N, 3, heads, hd)
    q, k, v = tok.permute(2, 0, 3, 1, 4)
    attn = (q * hd ** -0.5) @ k.transpose(-2, -1)
    table, index = dsd[bp + "attn.relative_position_bias_table"], dsd[bp + "attn.relative_position_index"]
    attn = attn + table[index].reshape(N, N, heads).permute(2, 0, 1).unsqueeze(0)
    if sh + sw > 0:
        diff = region.unsqueeze(1) != region.unsqueeze(2)
        mask = torch.where(diff, -100.0, 0.0).to(attn.dtype)
        attn = (attn.reshape(B, nW, heads, N, N) + mask[None, :, None]).reshape(B * nW, heads, N, N)
    ctx = (attn.softmax(-1) @ v).transpose(1, 2).reshape(B, nW * N, C_)
    res = qkv.new_zeros(B, H * W, C_)
    vf = valid.reshape(-1)
    res[:, src.reshape(-1)[vf], :] = ctx[:, vf, :]
    return res.reshape(B, H, W, C_)


@pytest.mark.parametrize("B,T,causal", [(10, 256, 0), (10, 100, 0), (3, 1, 0), (2, 77, 0), (1, 64, 0), (4, 150, 1), (2, 33, 1)])
def test_self_attention_matches_torch(B, T, causal):
    """hmocr_self_attention (tensor-core kernel when not causal) vs fp32 softmax(q k^T / sqrt(32)) v."""
    torch.manual_seed(B * 1000 + T)
    nhead, hd = 8, 32
    d = nhead * hd
    qkv = (torch.randn(B * T, 3 * d, device="cuda") * 1.5).half()
    ctx = torch.empty(B * T, d, device="cuda", dtype=torch.float16)
    lib, L = _lib()
    L.check(lib.hmocr_self_attention(P(qkv), B, T, nhead, causal, P(ctx), S()), "hmocr_self_attention")
    torch.cuda.synchronize()
    q, k, v = (x.float().view(B, T, nhead, hd).transpose(1, 2) for x in qkv.split(d, dim=1))
    sc = (q @ k.transpose(-1, -2)) / hd ** 0.5
    if causal:
        sc = sc + torch.full((T, T), float("-inf"), device="cuda").triu(1)
    ref = (sc.softmax(-1) @ v).transpose(1, 2).reshape(B * T, d)
    err = (ctx.float() - ref).abs().max().item()
    assert err < 4e-3, err


def test_gelu_epilogue_is_the_exact_erf_form_over_a_dense_grid():
    """nn.GELU() (erf form, swin_transformer.py:444) through the GEMM epilogue with an identity weight: the
    single-MUFU evaluation max(x,0) - |x| 2^q(|x|) stays within 2e-6 of x * Phi(x) on 16k points of [-9, 9]
    (fp32 output path), and the packed FFMA2 path of the fp16-output epilogue within one fp16 ulp of the exact value."""
    n = 64
    x = torch.linspace(-9.0, 9.0, 256 * n, device="cuda").half().view(256, n)       # exactly representable inputs
    w = torch.eye(n, device="cuda").half()
    ref = torch.nn.functional.gelu(x.double()).float()
    o32, _ = gemm(x, w, act=1, out_f32=True)
    assert (o32 - ref).abs().max().item() < 2e-6
    small = x.float().abs() < 1
    rel = ((o32 - ref).abs() / ref.abs().clamp_min(1e-30))[small & (ref != 0)]
    assert rel.max().item() < 2e-5
    _, o16 = gemm(x, w, act=1, out_f32=False, out_f16=True)
    assert torch.equal(o16, ref.half()) or (o16.float() - ref).abs().max().item() < 1e-3 * 9
    ulp_off = (o16.view(torch.int16).int() - ref.half().view(torch.int16).int()).abs().max().item()
    assert ulp_off <= 1, ulp_off


@pytest.mark.parametrize("M,K,N,fb", [(256, 64, 192, 2192), (300, 384, 1152, 2192), (1024, 1536, 384, 2192),
                                      (768, 768, 768, 2256), (515, 384, 1536, 2256), (7680, 3072, 768, 2192)])
def test_cta_pair_gemm_is_bit_identical_to_the_single_cta_kernel(M, K, N, fb):
    """cta_group::2 kernel (256-row tiles shared by two CTAs; force_bn 2192 / 2256 select it explicitly, K >= 1024
    shapes get it automatically) against the 1-CTA kernel: same MMA order along K, so the same bits - with the
    GELU fp16 epilogue and with the fp32 residual epilogue, ragged M included."""
    torch.manual_seed(M + K + N)
    a = torch.randn(M, K, device="cuda").half()
    w = (torch.randn(N, K, device="cuda") / K ** 0.5).half()
    b = torch.randn(N, device="cuda")
    r = torch.randn(M, N, device="cuda")
    one = 192 if fb == 2192 else 256
    _, p16 = gemm(a, w, bias=b, act=1, out_f32=False, out_f16=True, force_bn=fb)
    _, s16 = gemm(a, w, bias=b, act=1, out_f32=False, out_f16=True, force_bn=one)
    assert torch.equal(p16, s16)
    p32, _ = gemm(a, w, bias=b, residual=r, force_bn=fb)
    s32, _ = gemm(a, w, bias=b, residual=r, force_bn=one)
    assert torch.equal(p32, s32)
    assert (p32 - gemm_ref(a, w, bias=b, residual=r)).abs().max().item() < 2e-2
