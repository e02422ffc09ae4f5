"""GPU: teacher-forced scoring (``model.score`` / ``hmocr_score``) - per-token log-probabilities, row scores and the
argmax from one pass whose vocabulary projection keeps log-sum-exp partials instead of logits.

Checked against the float64 definition (tests/score_oracle.py::score_sequences) at every geometry of
tests/test_decode_geometry_gpu.py, against the engine's own ``decoder`` (which isolates the new epilogue and its
combine from the layer stack), at exact logit ties, against the decode paths it must agree with, and on its contract.
Lines starting with ``SCORE`` report the worst measured value of each check."""
import ctypes as C

import pytest
import torch

from test_decode_geometry_gpu import (BEAM_SCORE_TOL, DECODE_LOGP_TOL, EOS, GEOMETRIES, PAD, SOS, TIE_MARGIN, _engine,
                                      _geometry, _greedy, _oracle_logits, _oracle_sd, _synth, _tie_bound)

pytestmark = pytest.mark.gpu

CONF_TOL = 5e-3              # confidence against predict's (tests/test_parity_gpu.py, tests/test_nbest_gpu.py)
SCORE_ROWS_MAX_POS = 40      # BEAM_SCORE_TOL is stated for sums of up to 40 steps (tests/test_nbest_gpu.py, max_len=40)


def _sequential_sum(lp):
    acc = torch.zeros(lp.shape[:-1], dtype=torch.float32, device=lp.device)
    for t in range(lp.shape[-1]):
        acc = acc + lp[..., t]
    return acc


def _scored_mask(tokens):
    """tokens [N, 1+T] -> bool [N, T]: positions up to and including the first eos among columns 1..T."""
    body = tokens[:, 1:]
    seen = torch.cumsum((body == EOS).int(), -1) - (body == EOS).int()
    return seen == 0


def _mixed_tokens(greedy_tok, V, seed):
    """The engine's greedy rows (likely sequences) with every other row replaced by random ids and an eos at a random
    column (unlikely sequences: a user's correction need not be what the model would say)."""
    tok = greedy_tok.clone()
    N, W = tok.shape
    g = torch.Generator().manual_seed(seed)
    lo = 3 if V > 3 else 0
    rnd = torch.randint(lo, V, (N, W), generator=g).to(tok.device)
    stop = torch.randint(1, W, (N,), generator=g).tolist()
    for r in range(1, N, 2):
        tok[r, 1:] = rnd[r, 1:]
        if V > EOS and r % 4 == 1:
            tok[r, stop[r]] = EOS
    tok[:, 0] = SOS
    return tok


def _oracle_score(g, enc, tokens, chunk=8):
    from score_oracle import score_sequences
    lp, sc, am = [], [], []
    for i in range(0, tokens.shape[0], chunk):
        a, b, c = score_sequences(enc[i:i + chunk].double(), tokens[i:i + chunk], g.dsd, g.cfg)
        lp.append(a), sc.append(b), am.append(c)
    return torch.cat(lp), torch.cat(sc), torch.cat(am)


def _check_against_oracle(name, g, enc, tokens):
    lp, sc, am = g.model.score(encoder_out=enc, tokens=tokens, return_argmax=True)
    o_lp, o_sc, _ = _oracle_score(g, enc, tokens)
    ref = _oracle_logits(g, enc, tokens)
    mask = _scored_mask(tokens)
    assert (lp[~mask] == 0).all() and (am[~mask] == PAD).all()
    lp_err = float((lp.double() - o_lp)[mask].abs().max())
    am_safe = torch.where(mask, am.long(), torch.zeros_like(am.long()))
    assert ((am_safe >= 0) & (am_safe < g.V)).all()
    gap = (ref.max(-1).values - ref.gather(-1, am_safe.unsqueeze(-1)).squeeze(-1))[mask]
    gap_max = float(gap.max())
    short = mask.sum(1) <= SCORE_ROWS_MAX_POS
    sc_err = float((sc.double() - o_sc)[short].abs().max()) if bool(short.any()) else 0.0
    print(f"SCORE oracle {name}: rows {tokens.shape[0]} T {tokens.shape[1] - 1}: worst |logprob - fp64| {lp_err:.2e} "
          f"(tol {DECODE_LOGP_TOL}), worst argmax gap {gap_max:.2e} (tol {_tie_bound(ref):.2e}), worst |score - fp64| "
          f"{sc_err:.2e} over {int(short.sum())} rows <= {SCORE_ROWS_MAX_POS} positions (tol {BEAM_SCORE_TOL})")
    assert lp_err <= DECODE_LOGP_TOL
    assert gap_max <= _tie_bound(ref)
    assert sc_err <= BEAM_SCORE_TOL
    return lp, sc, am


# ---- 1. against the float64 definition ---------------------------------------------------------------------------
@pytest.mark.parametrize("geo", list(GEOMETRIES))
def test_score_against_fp64_oracle(geo):
    """Seeded features at every geometry of the decode tests (V = 5 .. 32771, L = 1 .. 12, max_seq_len up to 256, the
    ResNet-18 variant), on the engine's greedy rows and on random rows, over the full max_seq_len positions."""
    g = _geometry(geo)
    tok, steps, _, _, _ = _greedy(g)
    _check_against_oracle(geo, g, g.feats, _mixed_tokens(tok, g.V, seed=g.V + g.T))


@pytest.fixture(scope="module")
def golden(sd, cfg, golden_src):
    from handwritten_math_ocr_api_b200 import FormulaRecognitionModel

    class G:
        pass
    g = G()
    g.model = FormulaRecognitionModel(cfg.vocab_size)
    g.model.load_state_dict(sd)
    g.model.eval()
    g.V, g.cfg = cfg.vocab_size, cfg
    g.dsd = _oracle_sd(sd)
    g.feats = torch.from_numpy(golden_src["features"]).cuda()
    return g


def test_score_against_fp64_oracle_on_golden_features(golden):
    g = golden
    tok, steps, _ = g.model.generate(encoder_out=g.feats, max_len=g.cfg.max_seq_len)
    _check_against_oracle("golden", g, g.feats, _mixed_tokens(tok, g.V, seed=5))


# ---- 2. against the engine's own teacher-forced decoder ------------------------------------------------------------
@pytest.mark.parametrize("geo", ["v100_l1_t32", "v1033_l2_t160", "v5075_l8_t256_noeos", "v32771_l12_t64", "v5_l8_t2",
                                 "v1025_l3_t40_res18"])
def test_score_against_the_engines_decoder(geo):
    """Same layer stack, so the only difference is the epilogue: log-probs within 1e-4 of the fp64 log_softmax of
    ``model.decoder``'s logits, the argmax equal to ``argmax(-1)`` wherever top-1 and top-2 differ by more than 1e-4,
    and the score bit-equal to the sequential fp32 sum of the log-probs."""
    g = _geometry(geo)
    tok, _, _, _, _ = _greedy(g)
    tokens = _mixed_tokens(tok, g.V, seed=11)
    lp, sc, am = g.model.score(encoder_out=g.feats, tokens=tokens, return_argmax=True)
    logits = g.model.decoder(g.feats, tokens[:, :-1]).double()
    want = torch.log_softmax(logits, -1).gather(-1, tokens[:, 1:].unsqueeze(-1)).squeeze(-1)
    mask = _scored_mask(tokens)
    err = float((lp.double() - want)[mask].abs().max())
    top2 = logits.topk(min(2, g.V), -1).values
    clear = mask & ((top2[..., 0] - top2[..., -1]) > 1e-4) if g.V > 1 else mask
    mism = int((am.long() != logits.argmax(-1))[clear].sum())
    print(f"SCORE decoder {geo}: worst |logprob - fp64 log_softmax(decoder)| {err:.2e} (tol 1e-4), argmax mismatches "
          f"{mism} of {int(clear.sum())} clear positions")
    assert err <= 1e-4
    assert mism == 0
    assert torch.equal(sc, _sequential_sum(lp))


# ---- 3. exact ties and the tail mask ---------------------------------------------------------------------------------
TIE_PLACES = {"31_32": lambda V: [31, 32], "255_256": lambda V: [255, 256], "last": lambda V: [V - 1],
              "first_last": lambda V: [0, V - 1]}
_TIE_MODELS = {}


def _tie_bias(V, cols):
    """Every real bias negative: most at -6, a group of 64 moderate columns (the scored targets) at -1 .. -1.5, the
    tied maximum at -0.25.  A pad column past V that escaped the mask is an exact logit 0: it would win the argmax and
    add exp(0) per column to the sum."""
    b = -6.0 - 0.25 * (torch.arange(V) % 3).double()
    group = sorted({(37 * i + 5) % V for i in range(64)} | {EOS})
    b[group] = -1.0 - 0.125 * (torch.arange(len(group)) % 5).double()
    b[cols] = -0.25
    return b.float(), group


@pytest.mark.parametrize("place", list(TIE_PLACES))
@pytest.mark.parametrize("V", [1033, 5075])
def test_exact_ties_and_tail_mask(V, place):
    cols = TIE_PLACES[place](V)
    if V not in _TIE_MODELS:
        sd = _synth(V, 2, 24, "swin")
        sd["decoder.fc_out.weight"] = torch.zeros(V, 256)
        _TIE_MODELS[V] = sd
    sd = dict(_TIE_MODELS[V])
    bias, group = _tie_bias(V, cols)
    sd["decoder.fc_out.bias"] = bias
    m = _engine(V, 2, 24, "swin", sd)
    gen = torch.Generator().manual_seed(V)
    targets = torch.tensor(group + cols)
    tokens = targets[torch.randint(0, len(targets), (9, 25), generator=gen)].cuda()
    tokens[:, 0] = SOS
    tokens[0, 5] = EOS
    feats = torch.randn(9, 30, 256, generator=gen).cuda()
    lp, sc, am = m.score(encoder_out=feats, tokens=tokens, return_argmax=True)
    mask = _scored_mask(tokens)
    want = torch.log_softmax(bias.double(), -1).cuda()[tokens[:, 1:]]
    err = float((lp.double() - want)[mask].abs().max())
    print(f"SCORE ties V={V} at {cols}: worst |logprob - fp64 log_softmax(bias)| {err:.2e} (tol 1e-6)")
    assert (am[mask] == min(cols)).all()
    assert err <= 1e-6
    assert torch.equal(sc, _sequential_sum(lp))
    del m


# ---- 4. round trip with decoding ----------------------------------------------------------------------------------------
def test_score_of_greedy_tokens_matches_generate(golden):
    g = golden
    tok, steps, lp_gen = g.model.generate(encoder_out=g.feats, max_len=g.cfg.max_seq_len, return_logprobs=True)
    lp, sc, am = g.model.score(encoder_out=g.feats, tokens=tok, return_argmax=True)
    mask = _scored_mask(tok)
    err = float((lp - lp_gen).abs()[mask].max())
    ref = _oracle_logits(g, g.feats, tok)
    top2 = ref.topk(2, -1).values
    margin = top2[..., 0] - top2[..., 1]
    differ = mask & (am.long() != tok[:, 1:])
    worst_margin = float(margin[differ].max()) if bool(differ.any()) else 0.0
    print(f"SCORE greedy round trip: {steps} steps, worst |score logprob - generate logprob| {err:.2e} "
          f"(tol {DECODE_LOGP_TOL}), {int(differ.sum())} argmax != emitted, at oracle margins <= {worst_margin:.2e}")
    assert err <= DECODE_LOGP_TOL
    assert worst_margin < TIE_MARGIN


def test_score_of_nbest_hypotheses_matches_their_scores(golden):
    g = golden
    tk, sk, lpk, steps = g.model.generate_nbest(encoder_out=g.feats, beam_size=3, max_len=40)
    B, K, W = tk.shape
    _, sc = g.model.score(encoder_out=g.feats.repeat_interleave(K, 0), tokens=tk.reshape(B * K, W))
    err = float((sc.reshape(B, K) - sk).abs().max())
    print(f"SCORE n-best round trip (beam 3, {steps} steps): worst |score - n-best score| {err:.2e} "
          f"(tol {BEAM_SCORE_TOL})")
    assert err <= BEAM_SCORE_TOL


# ---- 5. contract details --------------------------------------------------------------------------------------------------
def test_eos_handling(golden):
    m, V = golden.model, golden.V
    feats = golden.feats
    gen = torch.Generator().manual_seed(3)
    tok = torch.randint(3, V, (4, 21), generator=gen).cuda()
    tok[:, 0] = SOS
    tok[0, 7] = EOS
    tok[1, 1] = EOS
    tok[3, 20] = EOS
    padded = tok.clone()
    padded[0, 8:] = PAD
    padded[1, 2:] = PAD
    garbage = tok.clone()
    garbage[0, 8:] = torch.randint(0, V, (13,), generator=gen).cuda()
    garbage[1, 2:] = EOS
    outs = [m.score(encoder_out=feats, tokens=t, return_argmax=True) for t in (tok, padded, garbage)]
    for o in outs[1:]:
        for a, b in zip(outs[0], o):
            assert torch.equal(a, b)
    lp, sc, am = outs[0]
    assert int((lp[1] != 0).sum()) == 1 and int((am[1] != PAD).sum()) == 1      # eos in column 1: one position
    assert int((am[0] != PAD).sum()) == 7 and (lp[0, 7:] == 0).all()
    assert bool((lp[2] != 0).all()) and bool((am[2] != PAD).all())             # no eos: all T positions
    assert torch.equal(sc, _sequential_sum(lp))
    # T = 1
    lp1, sc1, am1 = m.score(encoder_out=feats, tokens=tok[:, :2], return_argmax=True)
    assert lp1.shape == (4, 1) and torch.equal(sc1, lp1[:, 0])
    logits = m.decoder(feats, tok[:, :1]).double()
    want = torch.log_softmax(logits, -1)[:, 0].gather(-1, tok[:, 1:2]).squeeze(-1)
    assert float((lp1[:, 0].double() - want).abs().max()) <= 1e-4


def test_results_do_not_depend_on_the_batch(golden):
    m = golden.model
    feats = torch.randn(300, 30, 256, generator=torch.Generator().manual_seed(8)).cuda()
    feats[:4] = golden.feats
    tok, _, _ = m.generate(encoder_out=feats[:45], max_len=60)
    tok = _mixed_tokens(tok, golden.V, seed=9)
    tok300 = tok.repeat(7, 1)[:300]
    big = m.score(encoder_out=feats[:300], tokens=tok300, return_argmax=True)
    mid = m.score(encoder_out=feats[:45], tokens=tok, return_argmax=True)
    for r in (0, 1, 3, 44):
        alone = m.score(encoder_out=feats[r:r + 1], tokens=tok[r:r + 1], return_argmax=True)
        for a, b, c in zip(alone, mid, big):
            assert torch.equal(a[0], b[r]) and torch.equal(a[0], c[r]), r
    again = m.score(encoder_out=feats[:45], tokens=tok, return_argmax=True)
    for a, b in zip(mid, again):
        assert torch.equal(a, b)


def test_images_form_equals_encoder_output_form(sd, cfg, golden):
    from oracle.synth import synth_images
    m = golden.model
    imgs = synth_images(5, seed=77).cuda()
    enc = m.encoder(imgs)
    tok, _, _ = m.generate(encoder_out=enc, max_len=30)
    want = m.score(encoder_out=enc, tokens=tok, return_argmax=True)
    for _ in range(3):                 # eager, then the captured encoder graph, then its replay
        got = m.score(imgs, tokens=tok, return_argmax=True)
        for a, b in zip(want, got):
            assert torch.equal(a, b)


def test_images_form_resnet18_uses_the_pos_table():
    from handwritten_math_ocr_api_b200.synthetic import synth_pos_table
    from oracle.synth import synth_images
    g = _geometry("v1025_l3_t40_res18")
    imgs = synth_images(6, seed=5).cuda()
    pt = synth_pos_table(256, seed=2)
    enc = g.model.encoder(imgs, pos_table=pt)
    tok, _, _ = g.model.generate(encoder_out=enc, max_len=g.T)
    want = g.model.score(encoder_out=enc, tokens=tok)
    got = g.model.score(imgs, tokens=tok, pos_table=pt)
    assert torch.equal(want[0], got[0]) and torch.equal(want[1], got[1])


def test_refusals(golden):
    from handwritten_math_ocr_api_b200 import _lib
    m, V, T = golden.model, golden.V, golden.cfg.max_seq_len
    feats = golden.feats
    tok = torch.full((4, 6), 3, dtype=torch.int64, device="cuda")
    with pytest.raises(ValueError):
        m.score(encoder_out=feats, tokens=tok[0])                     # not [B, 1+T]
    with pytest.raises(ValueError):
        m.score(encoder_out=feats, tokens=tok[:3])                    # batch mismatch
    with pytest.raises(ValueError):
        m.score(tokens=tok)                                           # no input
    with pytest.raises(ValueError):
        m.score(encoder_out=feats[:, :10], tokens=tok)                # wrong memory shape
    bad = tok.clone()
    bad[1, 3] = V
    with pytest.raises(IndexError):
        m.score(encoder_out=feats, tokens=bad)
    bad[1, 3] = -1
    with pytest.raises(IndexError):
        m.score(encoder_out=feats, tokens=bad)
    with pytest.raises(RuntimeError):
        m.score(encoder_out=feats, tokens=tok[:, :1])                 # T = 0
    with pytest.raises(RuntimeError):
        m.score(encoder_out=feats, tokens=torch.full((4, T + 2), 3, dtype=torch.int64, device="cuda"))
    lib = _lib.load()
    rc = lib.hmocr_score(m._handle(), C.c_void_p(feats.data_ptr()), 1, 4, 5, C.c_void_p(tok.data_ptr()), None, None,
                         None, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc != 0 and b"NULL" in lib.hmocr_last_error()


# ---- 6. memory -----------------------------------------------------------------------------------------------------------
def _peak(fn):
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def test_score_allocates_no_logits(sd, cfg):
    """Fresh models at B = 256, T = 150 (each route sizes its own workspace): the peak of ``score`` stays at least one
    [B, T, V] fp32 tensor below the peak of decoder + log_softmax + gather."""
    from handwritten_math_ocr_api_b200 import FormulaRecognitionModel
    B, T, V = 256, 150, cfg.vocab_size
    gen = torch.Generator().manual_seed(1)
    feats = torch.randn(B, 30, 256, generator=gen).cuda()
    tok = torch.randint(3, V, (B, T + 1), generator=gen).cuda()
    tok[:, 0] = SOS

    def fresh():
        m = FormulaRecognitionModel(V)
        m.load_state_dict(sd)
        return m

    def torch_route(m):
        logits = m.decoder(feats, tok[:, :-1])
        torch.log_softmax(logits, -1).gather(-1, tok[:, 1:].unsqueeze(-1))

    m = fresh()
    p_score = _peak(lambda: m.score(encoder_out=feats, tokens=tok))
    del m
    m = fresh()
    p_dec = _peak(lambda: torch_route(m))
    del m
    torch.cuda.empty_cache()
    need = B * T * V * 4
    print(f"SCORE memory B={B} T={T}: peak score {p_score / 2**30:.3f} GiB, decoder+log_softmax+gather "
          f"{p_dec / 2**30:.3f} GiB, difference {(p_dec - p_score) / need:.2f} x B*T*V*4")
    assert p_dec - p_score >= need


# ---- 7. score_formulas on the golden images --------------------------------------------------------------------------
def test_score_formulas_reproduces_predict_confidence(sd, cfg, golden, golden_src):
    from handwritten_math_ocr_api_b200 import im2latex, inference
    from handwritten_math_ocr_api_b200.synthetic import synth_images, synth_vocab
    vocab, idx2char = synth_vocab(cfg.vocab_size)
    m = golden.model
    imgs = synth_images(2, int(golden_src["images_seed"])).cuda()
    preds = im2latex.predict_batch(m, imgs, vocab, idx2char, "cuda")
    tok, _, _ = m.generate(imgs, max_len=cfg.max_seq_len)
    raw = inference.ids_to_strings(tok.tolist(), idx2char)
    fits = [i for i, f in enumerate(raw) if len(f.split()) <= cfg.max_seq_len - 1]
    assert fits, "no golden image ends with eos"
    got = im2latex.score_formulas(m, imgs[fits], [raw[i] for i in fits], vocab, idx2char)
    for j, i in enumerate(fits):
        print(f"SCORE score_formulas image {i}: confidence {got[j][0]:.6f} vs predict {preds[i][1]:.6f}, "
              f"score {got[j][1]:.4f}")
        assert abs(got[j][0] - preds[i][1]) <= CONF_TOL
    for i in set(range(2)) - set(fits):              # a formula that never emitted eos cannot take one
        with pytest.raises(ValueError, match="max_seq_len"):
            im2latex.score_formulas(m, imgs[i:i + 1], [raw[i]], vocab, idx2char)
