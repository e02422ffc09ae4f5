"""GPU: n-best beam search (``generate_nbest`` / ``hmocr_generate_nbest``) - ranked hypotheses with per-token
log-probabilities, against ``generate(beam_size=K)``, the oracle, and itself (launch boundaries, batch composition,
repetition).  Definition of the search: oracle/decode.py::beam_search."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DECODE_LOGP_TOL = 1.5e-2      # per-token |log p - oracle| on identical encoder features (tests/test_model_gpu.py)
BEAM_SCORE_TOL = 5e-2         # |score - oracle score| of the best hypothesis (tests/test_model_gpu.py)
CONF_TOL = 5e-3               # confidence against the oracle's log-probs (tests/test_parity_gpu.py)


@pytest.fixture(scope="module")
def model(sd, cfg):
    from handwritten_math_ocr_api_b200 import FormulaRecognitionModel
    m = FormulaRecognitionModel(cfg.vocab_size)
    m.load_state_dict(sd)
    return m.eval()


@pytest.fixture(scope="module")
def gfeats(golden_src):
    return torch.from_numpy(golden_src["features"]).cuda()


@pytest.fixture(scope="module")
def feats45(model):
    from oracle.synth import synth_images
    imgs = synth_images(8, seed=99).cuda().repeat(6, 1, 1, 1)[:45].contiguous()
    return model.encoder(imgs).clone()


@pytest.fixture(scope="module")
def feats64(model):
    from oracle.synth import synth_images
    return model.encoder(synth_images(64, seed=321).cuda()).clone()


def _first_eos_mask(tokens, eos):
    """[..., 1+steps] tokens -> bool [..., steps]: True at every step after the hypothesis' first eos."""
    body = tokens[..., 1:]
    seen = torch.cumsum((body == eos).int(), -1)
    return (seen - (body == eos).int()) > 0


def _sequential_sum(lp):
    acc = torch.zeros(lp.shape[:-1], dtype=torch.float32, device=lp.device)
    for t in range(lp.shape[-1]):
        acc = acc + lp[..., t]
    return acc


def _check_rank0_and_sums(m, cfg, K, **src):
    tok, steps, _, score = m.generate(beam_size=K, max_len=40, **src)
    t1, s1, lp1, n1 = m.generate_nbest(beam_size=K, n_best=1, max_len=40, **src)
    tk, sk, lpk, nk = m.generate_nbest(beam_size=K, max_len=40, **src)
    assert n1 == nk == steps and tk.shape == (tok.shape[0], K, steps + 1) and lpk.shape == (tok.shape[0], K, steps)
    for t, s in ((t1, s1), (tk, sk)):
        assert torch.equal(t[:, 0], tok) and torch.equal(s[:, 0], score)
    for t, s, lp in ((t1, s1, lp1), (tk, sk, lpk)):
        assert torch.equal(_sequential_sum(lp), s)                      # scores are the recorded log-probs' sum
        after = _first_eos_mask(t, cfg.eos)
        assert (lp[after] == 0).all() and (t[..., 1:][after] == cfg.pad).all()
    return tk, sk, lpk


# ---- 1, 2: rank 0 is generate(beam_size=K); scores are sums of the recorded log-probs ------------------------------
@pytest.mark.parametrize("K", [2, 3, 5])
def test_rank0_is_generate_and_scores_are_sums(model, cfg, gfeats, feats45, K):
    _check_rank0_and_sums(model, cfg, K, encoder_out=gfeats)
    _check_rank0_and_sums(model, cfg, K, encoder_out=feats45)          # full and partial clusters


# ---- 3, 4: per-token values and the ranked list against the oracle ---------------------------------------------------
@pytest.mark.parametrize("K", [2, 3, 5])
def test_nbest_against_the_oracle(model, sd, cfg, gfeats, K):
    from oracle import decode as odec
    from oracle.ref_model import decoder_forward
    feats = gfeats[:3]
    tok, sc, lp, steps = model.generate_nbest(encoder_out=feats, beam_size=K, max_len=40)
    B = feats.shape[0]
    # 4: ranked, pairwise distinct
    assert (sc[:, 1:] <= sc[:, :-1]).all()
    for b in range(B):
        rows = {tuple(tok[b, j].tolist()) for j in range(K)}
        assert len(rows) == K
    # 3: every returned token's log-prob against the oracle's teacher-forced log_softmax
    enc = feats.cpu().repeat_interleave(K, 0)
    flat = tok.reshape(B * K, -1).cpu()
    with torch.no_grad():
        lsm = torch.log_softmax(decoder_forward(enc, flat[:, :-1], sd, cfg).float(), -1)
    want = lsm.gather(-1, flat[:, 1:].unsqueeze(-1)).squeeze(-1)
    live = ~_first_eos_mask(flat, cfg.eos)
    err = (want - lp.reshape(B * K, -1).cpu())[live].abs().max().item()
    print(f"beam {K}: max per-token |log p - oracle| {err:.2e}")
    assert err <= DECODE_LOGP_TOL
    # 4: the j-th best score against the oracle's j-th best (lower ranks may differ in path at near-ties)
    _, _, o_all, o_sc = odec.beam_search(feats.cpu(), sd, cfg, beam=K, max_len=40)
    order = torch.sort(o_sc, dim=-1, descending=True, stable=True).indices
    o_sorted = torch.gather(o_sc, 1, order)
    d = (sc.cpu() - o_sorted).abs().max().item()
    same = 0
    for b in range(B):
        for j in range(K):
            o = o_all[b, int(order[b, j])].tolist()
            n = min(len(o), tok.shape[2])
            same += int(o[:n] == tok[b, j, :n].tolist())
    print(f"beam {K}: max |score_j - oracle score_j| {d:.2e}; identical hypotheses {same}/{B * K}")
    assert d <= BEAM_SCORE_TOL


# ---- 5, 6: launch boundaries, batch invariance, repeatability at full occupancy ---------------------------------------
def _nbest64(model, feats, **kw):
    t, s, lp, n = model.generate_nbest(encoder_out=feats, beam_size=5, max_len=70, **kw)
    return t.clone(), s.clone(), lp.clone(), n


def _same_prefix(a, b, fill):
    """Equal on the shorter length; the longer one holds only `fill` beyond it."""
    n = min(a.shape[-1], b.shape[-1])
    longer = a if a.shape[-1] > b.shape[-1] else b
    return torch.equal(a[..., :n], b[..., :n]) and bool((longer[..., n:] == fill).all())


def test_two_waves_and_launch_boundaries_are_invisible(model, cfg, feats64):
    runs = [_nbest64(model, feats64)]
    model.set_option("steps_per_launch", 8)
    try:
        runs.append(_nbest64(model, feats64))
    finally:
        model.set_option("steps_per_launch", 0)
    for i in range(feats64.shape[0]):
        t1, s1, lp1, _ = _nbest64(model, feats64[i:i + 1])
        for t, s, lp, _ in runs:
            assert torch.equal(s[i], s1[0]), i
            assert _same_prefix(t[i], t1[0], cfg.pad) and _same_prefix(lp[i], lp1[0], 0.0), i


def test_repeatable_at_full_occupancy(model, feats64):
    ref = _nbest64(model, feats64)
    for _ in range(2):
        cur = _nbest64(model, feats64)
        assert cur[3] == ref[3]
        for a, b in zip(cur[:3], ref[:3]):
            assert torch.equal(a, b)


# ---- 7: beam 1 is greedy ----------------------------------------------------------------------------------------
def test_beam_one_is_greedy(model, cfg, gfeats, feats45):
    for feats in (gfeats, feats45):
        g_tok, g_steps, g_lp = model.generate(encoder_out=feats, max_len=48, return_logprobs=True)
        tok, sc, lp, steps = model.generate_nbest(encoder_out=feats, beam_size=1, max_len=48)
        assert steps == g_steps and tok.shape == (feats.shape[0], 1, steps + 1)
        worst = 0.0
        for r in range(feats.shape[0]):
            row = g_tok[r].tolist()
            n = row.index(cfg.eos) + 1 if cfg.eos in row else len(row)
            assert tok[r, 0, :n].tolist() == row[:n]
            assert (tok[r, 0, n:] == cfg.pad).all() and (lp[r, 0, n - 1:] == 0).all()
            worst = max(worst, (lp[r, 0, :n - 1] - g_lp[r, :n - 1]).abs().max().item())
        print(f"beam 1 vs greedy: max |log p| difference {worst:.2e}")
        assert worst <= 1e-4


# ---- 8: ResNet-18 variant ----------------------------------------------------------------------------------------
def test_res18_variant(cfg):
    import os
    from handwritten_math_ocr_api_b200.model_res18trans import FormulaRecognitionModel
    from handwritten_math_ocr_api_b200.synthetic import synth_images, synth_state_dict_res18
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "res18_golden.npz"))
    m = FormulaRecognitionModel(cfg.vocab_size)
    m.load_state_dict(synth_state_dict_res18(cfg, seed=0))
    pos = torch.from_numpy(gold["pos_table"])
    imgs = synth_images(4, int(gold["images_seed"])).cuda()
    feats = m.encoder(imgs, pos).clone()
    for K in (2, 3, 5):
        _check_rank0_and_sums(m, cfg, K, encoder_out=feats)
    # from images: generate_nbest sets the same pinned table that generate does
    tok, _, _, score = m.generate(imgs, max_len=40, beam_size=3, pos_table=pos)
    t, s, _, _ = m.generate_nbest(imgs, beam_size=3, max_len=40, pos_table=pos)
    assert torch.equal(t[:, 0], tok) and torch.equal(s[:, 0], score)


# ---- 9: argument checks, caller-owned workspace, the raw C ABI --------------------------------------------------
def test_argument_checks(model, gfeats):
    with pytest.raises(RuntimeError, match="n_best=0 outside"):
        model.generate_nbest(encoder_out=gfeats, beam_size=3, n_best=0, max_len=8)
    with pytest.raises(RuntimeError, match="n_best=4 outside"):
        model.generate_nbest(encoder_out=gfeats, beam_size=3, n_best=4, max_len=8)
    with pytest.raises(RuntimeError, match="beam=6 outside"):
        model.generate_nbest(encoder_out=gfeats, beam_size=6, n_best=1, max_len=8)


def test_caller_owned_workspace_and_full_width_outputs(sd, cfg, model, gfeats):
    """A fresh engine given only a workspace of hmocr_workspace_bytes(B, T, -beam) runs hmocr_generate_nbest (beam 1
    needs the beam buffers, which the greedy plan does not have); columns past `steps` are pad / 0."""
    from handwritten_math_ocr_api_b200 import FormulaRecognitionModel, _lib
    m = FormulaRecognitionModel(cfg.vocab_size)
    m.load_state_dict(sd)
    lib, h = m._eng.lib, m._handle()
    B, T = gfeats.shape[0], 40
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    keep = []
    for K in (1, 3):
        n = C.c_size_t()
        _lib.check(lib.hmocr_workspace_bytes(h, B, T, -K, C.byref(n)), "hmocr_workspace_bytes")
        ws = torch.empty(n.value, dtype=torch.uint8, device="cuda")
        keep.append(ws)
        _lib.check(lib.hmocr_set_workspace(h, C.c_void_p(ws.data_ptr()), n.value, stream), "hmocr_set_workspace")
        tok = torch.full((B, K, T + 1), -7, dtype=torch.int64, device="cuda")
        lp = torch.full((B, K, T), 7.0, device="cuda")
        sc = torch.empty(B, K, device="cuda")
        steps = torch.zeros(1, dtype=torch.int32, device="cuda")
        _lib.check(lib.hmocr_generate_nbest(h, C.c_void_p(gfeats.data_ptr()), 1, B, T, K, K, C.c_void_p(tok.data_ptr()),
                                            C.c_void_p(lp.data_ptr()), C.c_void_p(sc.data_ptr()),
                                            C.c_void_p(steps.data_ptr()), stream), "hmocr_generate_nbest")
        torch.cuda.synchronize()
        s = int(steps.item())
        assert (tok[:, :, 0] == cfg.sos).all() and (tok[:, :, s + 1:] == cfg.pad).all() and (lp[:, :, s:] == 0).all()
        t2, s2, lp2, n2 = model.generate_nbest(encoder_out=gfeats, beam_size=K, max_len=T)
        assert n2 == s and torch.equal(tok[:, :, : s + 1], t2) and torch.equal(sc, s2) and torch.equal(lp[:, :, :s], lp2)
    _lib.check(lib.hmocr_set_workspace(h, None, 0, stream), "hmocr_set_workspace")
    torch.cuda.synchronize()


# ---- 10: the API mirror ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [3, 5])
def test_predict_nbest(model, sd, cfg, golden_src, K):
    from handwritten_math_ocr_api_b200 import im2latex
    from handwritten_math_ocr_api_b200.synthetic import synth_vocab
    from oracle.ref_model import decoder_forward
    from oracle.synth import synth_images
    vocab, idx2char = synth_vocab(cfg.vocab_size)
    imgs = synth_images(4, int(golden_src["images_seed"])).cuda()
    got = im2latex.predict_nbest(model, imgs, vocab, idx2char, "cuda", beam_size=K, n_best=K)
    top = im2latex.predict_batch(model, imgs, vocab, idx2char, "cuda", beam_size=K)
    assert [g[0][:2] for g in got] == top
    assert im2latex.predict(model, imgs[:1], vocab, idx2char, "cuda", beam_size=K) == top[0]
    for hyps in got:
        assert len({f for f, _, _ in hyps}) == len(hyps) and [s for _, _, s in hyps] == sorted([s for _, _, s in hyps], reverse=True)
    # confidences against the same bookkeeping on the oracle's log-probs of the same hypotheses
    feats = model.encoder(imgs).cpu()
    tok, sc, _, _ = model.generate_nbest(imgs, beam_size=K, n_best=K, max_len=im2latex.config.max_seq_len)
    B = tok.shape[0]
    flat = tok.reshape(B * K, -1).cpu()
    with torch.no_grad():
        lsm = torch.log_softmax(decoder_forward(feats.repeat_interleave(K, 0), flat[:, :-1], sd, cfg).float(), -1)
    olp = lsm.gather(-1, flat[:, 1:].unsqueeze(-1)).squeeze(-1).reshape(B, K, -1)
    worst = 0.0
    for b in range(B):
        want = im2latex.rank_hypotheses(tok[b, :, 1:].tolist(), olp[b].tolist(), sc[b].tolist(), vocab["<eos>"], idx2char)
        assert [w[0] for w in want] == [g[0] for g in got[b]]
        for (_, cw, _), (_, cg, _) in zip(want, got[b]):
            worst = max(worst, abs(cw - cg))
    print(f"beam {K}: max |confidence - oracle bookkeeping| {worst:.2e}")
    assert worst <= CONF_TOL
