"""GPU: the persistent decode kernel at every model geometry the engine accepts, against a float64 oracle.

The kernel's launch parameters come from the checkpoint's geometry: the vocabulary V sets the fc_out tiles per CTA
(``round_up(ceil(V / 128), 8)``), the slice of columns each of the 8 CTAs owns and the half-tile masks at the tail;
the layer count L sets the period of the weight stream (``20 L + fc_tiles`` chunks, so the warp that owns the first
fc_out tile moves from step to step when L is odd); max_seq_len sets the number of 32-key cache blocks and which
build runs (5 blocks up to 160 positions, 8 above).  Each row of ``GEOMETRIES`` exists for the edge it reaches.

Every check is made on the engine's OWN tokens: the float64 oracle (oracle/ref_model.py) is run teacher-forced on
the emitted prefix, so every emitted step of every row is checked, not only the part before a first divergence.
The exact-tie tests zero ``fc_out.weight``: every logit is then exactly its bias, whatever the summation order,
and the expected tokens follow from the tie rules alone (greedy: lowest index; beam: lower ``hyp * V + token``;
finalize: lower beam index).
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

TIE_MARGIN = 2e-2          # a chosen token's fp64 logit may trail the maximum by this much (tests/test_parity_gpu.py)
DECODE_LOGP_TOL = 1.5e-2   # per-step |log p - fp64 log_softmax| (tests/test_parity_gpu.py)
LOGIT_TOL = 1.5e-2         # teacher-forced logits, every vocabulary column (tests/test_parity_gpu.py)
BEAM_SCORE_TOL = 5e-2      # best beam score against the fp64 beam search (tests/test_nbest_gpu.py)
GREEDY_ROWS = 45           # 5 full 8-row clusters and one partial
BEAM_IMAGES = 13
WALK_GAIN = 24.0
SOS, EOS, PAD = 1, 2, 0

# name: (V, L, max_seq_len, encoder, eos_bias_sigma)
GEOMETRIES = {
    "v100_l1_t32": (100, 1, 32, "swin", 2.5),           # CTAs 1-7 hold no valid column; one cache block; one layer
    "v1025_l3_t33": (1025, 3, 33, "swin", 2.5),         # 16 tiles per CTA, column 1024 alone in CTA 4; odd L; 2nd block
    "v1033_l2_t160": (1033, 2, 160, "swin", 2.5),       # tail ends 1 column past a half-tile; longest 5-block build
    "v5075_l8_t161": (5075, 8, 161, "swin", 2.5),       # 8-block build with 6 cache blocks
    "v5075_l8_t256_noeos": (5075, 8, 256, "swin", 0.0),  # beam search past step 160 (8-block beam build)
    "v32771_l12_t64": (32771, 12, 64, "swin", 2.5),     # 264 fc tiles per CTA; L > 8
    "v5_l8_t2": (5, 8, 2, "swin", 2.5),                 # smallest max_seq_len; V equals the largest beam
    "v1025_l3_t40_res18": (1025, 3, 40, "res18", 2.5),  # the ResNet-18 variant (10 memory tokens)
}


def fc_tiles(V):
    return (-(-V // 128) + 7) // 8 * 8


def _model_config(V, L, T):
    from oracle.arch import ModelConfig
    return ModelConfig(vocab_size=V, num_layers=L, max_seq_len=T)


def _engine(V, L, T, arch, sd):
    from handwritten_math_ocr_api_b200.config import Config

    class C(Config):
        swin_num_decoder_layers = L
        num_decoder_layers = L
        res18trans_num_decoder_layers = L
        res18trans_num_encoder_layers = L      # synth_state_dict_res18 gives the encoder as many layers
        max_seq_len = T

    if arch == "res18":
        from handwritten_math_ocr_api_b200.model_res18trans import FormulaRecognitionModel
    else:
        from handwritten_math_ocr_api_b200 import FormulaRecognitionModel
    m = FormulaRecognitionModel(V, config=C())
    m.load_state_dict(sd)
    return m.eval()


def _synth(V, L, T, arch, **kw):
    from handwritten_math_ocr_api_b200.synthetic import synth_state_dict, synth_state_dict_res18
    cfg = _model_config(V, L, T)
    return (synth_state_dict_res18 if arch == "res18" else synth_state_dict)(cfg, seed=0, **kw)


def _oracle_sd(sd):
    """fp64 decoder weights on the GPU, under the Swin decoder's key names (the oracle's)."""
    return {k.replace("decoder.transformer_decoder.", "decoder.decoder."): v.to("cuda", torch.float64)
            for k, v in sd.items() if k.startswith("decoder.")}


def _feats(n, mem_tokens, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, mem_tokens, 256, generator=g).cuda()


class Geo:
    pass


_CACHE = {}


def _geometry(name):
    if name not in _CACHE:
        V, L, T, arch, eos_sigma = GEOMETRIES[name]
        g = Geo()
        g.V, g.L, g.T, g.arch = V, L, T, arch
        g.cfg = _model_config(V, L, T)
        sd = _synth(V, L, T, arch, eos_bias_sigma=eos_sigma)
        g.model = _engine(V, L, T, arch, sd)
        g.dsd = _oracle_sd(sd)
        g.feats = _feats(GREEDY_ROWS, g.model.mem_tokens, seed=V * 1000 + L * 100 + T)
        g.greedy = None
        g.eos_free = eos_sigma == 0
        _CACHE[name] = g
    return _CACHE[name]


def _oracle_logits(g, enc, tokens, chunk=8):
    """fp64 logits [N, n, V] of the oracle teacher-forced on tokens[:, :n] (tokens [N, 1+n])."""
    from oracle.ref_model import decoder_forward
    out = []
    with torch.no_grad():
        for i in range(0, tokens.shape[0], chunk):
            out.append(decoder_forward(enc[i:i + chunk].double(), tokens[i:i + chunk, :-1], g.dsd, g.cfg))
    return torch.cat(out)


def _tie_bound(ref):
    # a near-tie scales with the logits: fp16 operands carry a relative error (tests/test_parity_gpu.py)
    return TIE_MARGIN * max(1.0, float(ref.abs().max()) / 20.0)


def _greedy(g):
    """The persistent greedy decode of the 45 rows and the oracle's fp64 logits on its tokens (cached)."""
    if g.greedy is None:
        tok, steps, lp = g.model.generate_device(encoder_out=g.feats, max_len=g.T, return_logprobs=True)
        steps = int(steps.item())
        ran = g.model.last_decode_steps()
        ref = _oracle_logits(g, g.feats, tok[:, : steps + 1])
        g.greedy = (tok.clone(), steps, lp.clone(), ran, ref)
    return g.greedy


def _first_eos(body):
    """body [N, n] -> 1-based step of each row's first eos, or 0 when it has none."""
    is_eos = body == EOS
    return torch.where(is_eos.any(1), is_eos.int().argmax(1) + 1, torch.zeros_like(body[:, 0]))


def _after_eos(tokens):
    """[..., 1+n] -> bool [..., n]: True at every step after the row's first eos."""
    body = tokens[..., 1:]
    seen = torch.cumsum((body == EOS).int(), -1)
    return (seen - (body == EOS).int()) > 0


def _nbest_beam1_full_width(m, feats, T):
    """``hmocr_generate_nbest`` at beam 1 into full-width outputs: tokens [B, 1+T], including the pad past ``steps``
    (``generate_nbest`` slices them off)."""
    import ctypes as C
    from handwritten_math_ocr_api_b200 import _lib
    B = feats.shape[0]
    m._reserve("nbest", B, T, 1)
    tok = torch.full((B, 1, T + 1), -7, dtype=torch.int64, device="cuda")
    steps = torch.zeros(1, dtype=torch.int32, device="cuda")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(m._eng.lib.hmocr_generate_nbest(m._handle(), C.c_void_p(feats.data_ptr()), 1, B, T, 1, 1,
                                                C.c_void_p(tok.data_ptr()), None, None, C.c_void_p(steps.data_ptr()),
                                                stream), "hmocr_generate_nbest")
    return tok[:, 0], int(steps.item())


def _sequential_sum(lp):
    acc = torch.zeros(lp.shape[:-1], dtype=torch.float32, device=lp.device)
    for t in range(lp.shape[-1]):
        acc = acc + lp[..., t]
    return acc


# ---- greedy ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("geo", list(GEOMETRIES))
def test_greedy_against_fp64_oracle(geo):
    """Every step of every row: the token is in range and within a near-tie of the fp64 argmax, its log-prob matches
    the fp64 log_softmax, ``steps`` follows the stopping rule, and the kernel left its loop at most 2 steps late."""
    g = _geometry(geo)
    tok, steps, lp, ran, ref = _greedy(g)
    T, V = g.T, g.V
    assert tok.shape == (GREEDY_ROWS, T + 1)
    assert (tok[:, 0] == SOS).all() and (tok[:, steps + 1:] == PAD).all()
    body = tok[:, 1: steps + 1]
    assert ((body >= 0) & (body < V)).all()
    first = _first_eos(body)
    assert steps == (int(first.max()) if bool((first > 0).all()) else T)
    assert steps <= ran <= steps + 2, (steps, ran)
    chosen = ref.gather(-1, body.unsqueeze(-1)).squeeze(-1)
    gap = float((ref.max(-1).values - chosen).max())
    want_lp = torch.log_softmax(ref, -1).gather(-1, body.unsqueeze(-1)).squeeze(-1)
    lp_err = float((lp[:, :steps].double() - want_lp).abs().max())
    print(f"{geo}: steps {steps} (ran {ran}), worst oracle gap {gap:.2e} (bound {_tie_bound(ref):.2e}), "
          f"worst per-step log-prob error {lp_err:.2e}")
    assert gap < _tie_bound(ref)
    assert lp_err < DECODE_LOGP_TOL


@pytest.mark.parametrize("geo", list(GEOMETRIES))
def test_teacher_forced_logits_every_column(geo):
    """``model.decoder`` on the greedy tokens against the fp64 logits in all V columns (vocabulary padding of the
    teacher-forced path and its logits copy)."""
    g = _geometry(geo)
    tok, steps, _, _, ref = _greedy(g)
    logits = g.model.decoder(g.feats, tok[:, :steps])
    assert logits.shape == (GREEDY_ROWS, steps, g.V)
    err = float((logits.double() - ref).abs().max())
    print(f"{geo}: teacher-forced max |logit - fp64| {err:.2e} over {steps} positions x {g.V} columns")
    assert err < LOGIT_TOL


@pytest.mark.parametrize("geo", list(GEOMETRIES))
def test_beam_one_nbest_and_scoring_reproduce_greedy(geo):
    """Beam-1 n-best (beam 1 through the beam build) is the greedy decode, padded after each row's eos.  Teacher-forced
    scoring of the greedy tokens (``hmocr_score``, which shares no code with the decode kernel) gives every scored
    position the decode's log-prob, and its argmax is the emitted token up to an fp64 near-tie."""
    g = _geometry(geo)
    m = g.model
    tok, steps, lp, _, ref = _greedy(g)
    tb, sb = _nbest_beam1_full_width(m, g.feats, g.T)
    want = tok.clone()
    want[:, 1:][_after_eos(tok)] = PAD
    assert sb == steps and torch.equal(tb, want)
    seq = tok[:, : steps + 1]
    lp_s, _, am = m.score(encoder_out=g.feats, tokens=seq, return_argmax=True)
    scored = ~_after_eos(seq)                     # up to and including each row's first eos
    body, am = seq[:, 1:], am.long()
    assert ((am >= 0) & (am < g.V))[scored].all()
    lp_err = float((lp_s - lp[:, :steps]).abs()[scored].max())
    differ = scored & (am != body)
    gap = (ref.gather(-1, am.unsqueeze(-1)) - ref.gather(-1, body.unsqueeze(-1))).squeeze(-1).abs()[differ]
    worst = float(gap.max()) if gap.numel() else 0.0
    print(f"{geo}: score vs generate over {int(scored.sum())} positions: worst log-prob difference {lp_err:.2e}, "
          f"argmax != emitted at {int(differ.sum())}, fp64 gaps there <= {worst:.2e} (bound {_tie_bound(ref):.2e})")
    assert lp_err < DECODE_LOGP_TOL
    assert worst < _tie_bound(ref)


# ---- beam search and n-best -----------------------------------------------------------------------------------------
def _check_beam_step(g, feats, K, t):
    """The engine's K hypotheses after step t + 1 are the K best expansions, by fp64 score, of its K hypotheses after
    step t (each a ``max_len`` = t call: the search does not depend on max_len).  A swap of two candidates is forgiven
    only when their fp64 scores are closer than the engine's own score error allows.  -> (worst score error, margin)"""
    m = g.model
    B = feats.shape[0]
    ha, sa, _, na = m.generate_nbest(encoder_out=feats, beam_size=K, max_len=t)
    hb, sb, _, nb = m.generate_nbest(encoder_out=feats, beam_size=K, max_len=t + 1)
    assert na == t and nb == t + 1
    flat = ha.reshape(B * K, t + 1)
    ref = _oracle_logits(g, feats.repeat_interleave(K, 0), torch.cat([flat, flat[:, :1]], 1))     # positions 0..t
    lsm = torch.log_softmax(ref, -1)
    after = _after_eos(flat)
    s64 = lsm[:, :t].gather(-1, flat[:, 1:].unsqueeze(-1)).squeeze(-1).masked_fill(after, 0.0).sum(-1)
    fin = (flat[:, 1:] == EOS).any(-1)
    cand = s64.unsqueeze(-1) + lsm[:, t]
    frozen = torch.full_like(cand, float("-inf"))
    frozen[:, PAD] = s64
    cand = torch.where(fin.unsqueeze(-1), frozen, cand).reshape(B, K, -1)
    err = float((sa.reshape(-1).double() - s64).abs().max())
    margin = 2 * err + DECODE_LOGP_TOL
    for b in range(B):
        chosen = torch.zeros_like(cand[b], dtype=torch.bool)
        for i in range(K):
            parent = [j for j in range(K) if torch.equal(ha[b, j], hb[b, i, : t + 1])]
            assert len(parent) == 1, (b, i)
            chosen[parent[0], int(hb[b, i, t + 1])] = True
            assert abs(float(sb[b, i]) - float(cand[b, parent[0], int(hb[b, i, t + 1])])) < margin, (b, i)
        assert int(chosen.sum()) == K
        assert float(cand[b][chosen].min()) > float(cand[b][~chosen].max()) - margin, (b, t)
    return err, margin


@pytest.mark.parametrize("K", [2, 5])
@pytest.mark.parametrize("geo", list(GEOMETRIES))
def test_beam_nbest_against_fp64_oracle(geo, K):
    """Rank 0 is ``generate(beam_size=K)``, scores are the fp32 sums of the per-token log-probs, every live per-token
    log-prob matches the fp64 log_softmax, and the selection of several steps (around step 160 and past it at 256
    positions) is checked against the fp64 scores of the engine's own hypotheses.  The best score is compared with
    the fp64 beam search where both searches return the same best hypothesis.  Over 256 steps of near-flat logits
    the two searches part at near-ties and then follow different paths: on a B200 they returned the same best
    hypothesis for 9 of 13 images at beam 2 and 10 of 13 at beam 5, and the best scores of the others differed by up
    to 23 and 143.  The per-step check above covers the selection there without depending on which side of a
    near-tie each search fell."""
    from oracle import decode as odec
    g = _geometry(geo)
    m, T, V = g.model, g.T, g.V
    feats = g.feats[:BEAM_IMAGES]
    tok, steps, _, score = m.generate(encoder_out=feats, beam_size=K, max_len=T)
    tk, sk, lpk, nk = m.generate_nbest(encoder_out=feats, beam_size=K, max_len=T)
    assert nk == steps and tk.shape == (BEAM_IMAGES, K, steps + 1)
    assert torch.equal(tk[:, 0], tok) and torch.equal(sk[:, 0], score)
    assert torch.equal(_sequential_sum(lpk), sk)
    assert (tk[..., 0] == SOS).all() and ((tk >= 0) & (tk < V)).all()
    after = _after_eos(tk)
    assert (lpk[after] == 0).all() and (tk[..., 1:][after] == PAD).all()
    assert (sk[:, 1:] <= sk[:, :-1]).all()
    if g.eos_free:
        assert steps > 160, steps                   # the 8-block beam build ran past the 5-block range
    flat = tk.reshape(BEAM_IMAGES * K, -1)
    ref = _oracle_logits(g, feats.repeat_interleave(K, 0), flat)
    want = torch.log_softmax(ref, -1).gather(-1, flat[:, 1:].unsqueeze(-1)).squeeze(-1)
    live = ~after.reshape(BEAM_IMAGES * K, -1)
    lp_err = float((lpk.reshape(BEAM_IMAGES * K, -1).double() - want)[live].abs().max())
    assert lp_err < DECODE_LOGP_TOL
    probe = {1, steps // 2, steps - 1} | ({159, 160, 161, 200, steps - 1} if steps > 160 else set())
    step_err = 0.0
    for t in sorted(x for x in probe if 1 <= x < steps):
        step_err = max(step_err, _check_beam_step(g, feats, K, t)[0])
    o_tok, o_best, _, _ = odec.beam_search(feats.double(), g.dsd, g.cfg, beam=K, max_len=T)
    same = [b for b in range(BEAM_IMAGES) if o_tok.shape[-1] == tk.shape[-1] and torch.equal(o_tok[b], tk[b, 0])]
    score_err = float((sk[same, 0].double() - o_best[same]).abs().max()) if same else 0.0
    print(f"{geo} beam {K}: steps {steps}, worst per-token log-prob error {lp_err:.2e}, worst hypothesis score error "
          f"{step_err:.2e}, same best hypothesis as the fp64 search on {len(same)}/{BEAM_IMAGES} images, "
          f"best score difference there {score_err:.2e}")
    assert score_err < BEAM_SCORE_TOL


# ---- a designed walk through the columns at slice and tile edges ----------------------------------------------------
def boundary_columns(V):
    """0, 7, 8, 15, 16, every CTA's first and last column below V, V-9, V-8 and V-1 (without sos / eos, once each)."""
    cpc = 16 * fc_tiles(V)
    cols = [0, 7, 8, 15, 16]
    for c in range(8):
        if c * cpc < V:
            cols += [c * cpc, min((c + 1) * cpc, V) - 1]
    cols += [V - 9, V - 8, V - 1]
    out = []
    for c in cols:
        if 0 <= c < V and c not in (SOS, EOS) and c not in out:
            out.append(c)
    return out


@pytest.mark.parametrize("geo", list(GEOMETRIES))
def test_designed_walk_through_boundary_columns(geo):
    """``fc_out.weight[next] += gain * unit(embedding[prev])`` chains sos -> c0 -> c1 -> ... through the boundary
    columns (the ``peak`` construction of synthetic.py with a chosen successor).  The fp64 oracle follows the chain
    (a check of the construction); the engine must emit it exactly, so a masking or merge error at a slice or tile
    edge shows as a wrong token, not inside a tolerance."""
    from oracle import decode as odec
    V, L, T, arch, _ = GEOMETRIES[geo]
    chain = boundary_columns(V)[:T]
    sd = _synth(V, L, T, arch, eos_bias_sigma=0.0)
    emb = sd["decoder.embedding.weight"].double()
    unit = emb / emb.norm(dim=1, keepdim=True)
    w = sd["decoder.fc_out.weight"].double()
    prev = SOS
    for c in chain:
        w[c] += WALK_GAIN * unit[prev]
        prev = c
    sd["decoder.fc_out.weight"] = w.float()
    m = _engine(V, L, T, arch, sd)
    feats = _feats(16, m.mem_tokens, seed=7 * V + L)
    n = len(chain)
    want = torch.tensor([SOS] + chain, device="cuda").expand(16, -1)
    g = Geo()
    g.dsd, g.cfg = _oracle_sd(sd), _model_config(V, L, T)
    ys = odec.greedy_cached(feats.double(), g.dsd, g.cfg, max_len=n)
    assert torch.equal(ys[:, : n + 1], want), "the construction does not steer the fp64 oracle: raise WALK_GAIN"
    tok, steps, _ = m.generate(encoder_out=feats, max_len=n)
    assert steps == n and torch.equal(tok, want)
    for K in (2, 5):
        tk, _, _, _ = m.generate(encoder_out=feats, beam_size=K, max_len=n)
        o_tok, _, _, _ = odec.beam_search(feats.double(), g.dsd, g.cfg, beam=K, max_len=n)
        assert torch.equal(tk, o_tok), K


# ---- exact ties -------------------------------------------------------------------------------------------------------
def _tie_groups(V):
    """Columns that tie: both halves of one 16-row tile (33, 41), tiles of other warps (53, 70), other CTAs, 0 and V-1."""
    cpc = 16 * fc_tiles(V)
    cols = [0, 33, 41, 53, 70] + [c * cpc + 3 * c for c in range(1, 8)] + [V - 1]
    return sorted({c for c in cols if 0 <= c < V and c not in (SOS, EOS)})


def _bias_spread(V):
    """Top group at -1 (below the 0 logit of the zero weight rows past V), eos and a few columns at -1.5, the rest -3."""
    b = torch.full((V,), -3.0)
    b[_tie_groups(V)] = -1.0
    b[[EOS, 4, 5]] = -1.5
    return b


def _bias_frozen(V):
    """One top token at 0, eos alone at -800, the rest at -1600.  exp(-800) underflows in fp32 AND fp64, so the
    log-sum-exp is exactly 0 in both and every log-prob is exactly its bias: a finished hypothesis' frozen score
    ties bit for bit with live candidates, and the tie rules alone decide."""
    b = torch.full((V,), -1600.0)
    b[V - 5] = 0.0
    b[EOS] = -800.0
    return b


TIE_CASES = [(V, kind) for V in (1025, 1033, 5075) for kind in ("spread", "frozen")]
_TIE_CACHE = {}


def _tie_engine(V, kind):
    if (V, kind) not in _TIE_CACHE:
        L, T = 2, 24
        sd = _synth(V, L, T, "swin")
        sd["decoder.fc_out.weight"] = torch.zeros(V, 256)
        sd["decoder.fc_out.bias"] = _bias_spread(V) if kind == "spread" else _bias_frozen(V)
        g = Geo()
        g.V, g.L, g.T = V, L, T
        g.model = _engine(V, L, T, "swin", sd)
        g.dsd, g.cfg = _oracle_sd(sd), _model_config(V, L, T)
        g.bias = sd["decoder.fc_out.bias"].double()
        g.feats = _feats(11, 30, seed=V + len(kind))
        _TIE_CACHE[(V, kind)] = g
    return _TIE_CACHE[(V, kind)]


@pytest.mark.parametrize("V,kind", TIE_CASES)
def test_exact_ties_greedy_in_decode_and_scoring(V, kind):
    """Greedy picks the lowest index of the maximum at every step (torch.argmax), on the persistent kernel and beam-1
    n-best, and its log-prob is log_softmax(bias)[token].  Teacher-forced scoring's argmax, a second arg-max
    implementation, gives the same token at every position with the same log-prob."""
    g = _tie_engine(V, kind)
    m, T = g.model, g.T
    top = int(torch.nonzero(g.bias == g.bias.max())[0])
    want_lp = float(torch.log_softmax(g.bias, -1)[top])
    want = torch.full((g.feats.shape[0], T + 1), top, device="cuda")
    want[:, 0] = SOS
    tok, steps, lp = m.generate(encoder_out=g.feats, max_len=T, return_logprobs=True)
    assert steps == T and torch.equal(tok, want)
    assert float((lp.double() - want_lp).abs().max()) < 1e-5
    lp_s, _, am = m.score(encoder_out=g.feats, tokens=want, return_argmax=True)
    assert torch.equal(am.long(), want[:, 1:])
    assert float((lp_s.double() - want_lp).abs().max()) < 1e-5
    tk, _, _, steps = m.generate_nbest(encoder_out=g.feats, beam_size=1, max_len=T)
    assert steps == T and torch.equal(tk[:, 0], want)


@pytest.mark.parametrize("K", [2, 3, 5])
@pytest.mark.parametrize("V,kind", TIE_CASES)
def test_exact_ties_beam_and_nbest(V, kind, K):
    """Every hypothesis, token for token, against the fp64 beam search on the same constant logits (ties -> lower
    ``hyp * V + token``), and the n-best ranking of equal final scores by lower beam index."""
    from oracle import decode as odec
    g = _tie_engine(V, kind)
    m, T = g.model, g.T
    feats = g.feats[:3]
    tk, sk, lpk, steps = m.generate_nbest(encoder_out=feats, beam_size=K, max_len=T)
    _, _, o_all, o_sc = odec.beam_search(feats.double(), g.dsd, g.cfg, beam=K, max_len=T)
    assert steps == o_all.shape[-1] - 1
    order = torch.sort(o_sc, dim=-1, descending=True, stable=True).indices
    o_tok = torch.gather(o_all, 1, order.unsqueeze(-1).expand(-1, -1, o_all.shape[-1]))
    o_sorted = torch.gather(o_sc, 1, order)
    assert torch.equal(tk, o_tok)
    # "frozen": every score is a sum of exact multiples of 800.  "spread": T fp32 additions of a log-prob near -5
    tol = 0.0 if kind == "frozen" else 1e-4 * T
    assert float((sk.double() - o_sorted).abs().max()) <= tol
    tok, s1, _, score = m.generate(encoder_out=feats, beam_size=K, max_len=T)
    assert s1 == steps and torch.equal(tok, tk[:, 0]) and torch.equal(score, sk[:, 0])
    if kind == "frozen":
        # equal final scores exist (several hypotheses at -800 * k): the lower beam index ranks first, as in the oracle
        assert bool((o_sorted[:, 1:] == o_sorted[:, :-1]).any()) or K == 2


# ---- fewer tokens than hypotheses --------------------------------------------------------------------------------------
def test_beam_wider_than_the_vocabulary_is_refused():
    """A beam keeps ``beam`` distinct tokens per hypothesis and step; V = 4 cannot fill beam 5 and the call fails with a
    message before anything runs.  beam 4 = V still decodes, against the fp64 beam search."""
    from oracle import decode as odec
    V, L, T = 4, 1, 8
    sd = _synth(V, L, T, "swin")
    m = _engine(V, L, T, "swin", sd)
    feats = _feats(3, 30, seed=4)
    with pytest.raises(RuntimeError, match="beam=5 exceeds vocab_size=4"):
        m.generate(encoder_out=feats, beam_size=5, max_len=T)
    with pytest.raises(RuntimeError, match="beam=5 exceeds vocab_size=4"):
        m.generate_nbest(encoder_out=feats, beam_size=5, max_len=T)
    tk, sk, _, steps = m.generate_nbest(encoder_out=feats, beam_size=4, max_len=T)
    assert ((tk >= 0) & (tk < V)).all() and steps >= 1
    _, o_best, _, _ = odec.beam_search(feats.double(), _oracle_sd(sd), _model_config(V, L, T), beam=4, max_len=T)
    assert float((sk[:, 0].double() - o_best).abs().max()) < BEAM_SCORE_TOL
