"""GPU parity of the engine (through the C ABI) against the golden vectors of the real reference
and against the oracle run on the same seeded inputs.

Stated tolerances (north_star: "within a stated bf16/fp32 tolerance ... e.g. max-abs logit error <= 1e-2"):
  * the engine computes in fp16 operands (saturating conversions), fp32 accumulation, fp32 residual stream /
    LayerNorm / softmax
  * encoder features (std ~1.2, |max| ~4): max-abs error <= 1e-2            (measured 3.7e-3)
  * teacher-forced logits (std ~4):        max-abs error <= 1e-2            (measured 7.8e-3)
  * greedy tokens: identical, or first divergence at a step whose reference top1-top2 margin is
    below 2x the logit tolerance (a near-tie, allowed by north_star; measured margins <= 3.2e-3).
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

FEAT_TOL = 1e-2
LOGIT_TOL = 1e-2
# the persistent decode kernel on identical encoder features: measured max |log p(winner) - oracle| 5.0e-3,
# largest oracle margin at a divergence 2.4e-3 (58/64 sequences of 60 steps identical)
DECODE_LOGP_TOL = 1.5e-2
DECODE_TIE_MARGIN = 1e-2


@pytest.fixture(scope="module")
def model(sd, cfg):
    from handwritten_math_ocr_api_b200 import FormulaRecognitionModel
    m = FormulaRecognitionModel(cfg.vocab_size)
    m.load_state_dict(sd)
    return m.eval()


@pytest.fixture(scope="module")
def dsd(sd):
    return {k: v.cuda() for k, v in sd.items()}


def _images(golden_src, n=4):
    from oracle.synth import synth_images
    return synth_images(n, int(golden_src["images_seed"]))


def test_param_count_and_surface(model):
    assert sum(p.numel() for p in model.parameters()) == 37_450_293      # README.md:89
    assert model.to("cuda") is model and model.eval() is model
    with pytest.raises(RuntimeError):
        model.to("cpu")


def test_encoder_against_reference_golden(model, golden_src):
    feats = model.encoder(_images(golden_src).cuda())
    assert feats.shape == (4, 30, 256) and feats.dtype == torch.float32
    err = np.abs(feats.cpu().numpy() - golden_src["features"]).max()
    print("encoder max-abs error vs reference:", err)
    assert err < FEAT_TOL


def test_encoder_is_batch_independent(model, golden_src):
    """Per-image features do not depend on batch-mates (SURVEY.md 8e): bit-identical at B=1 and B=3."""
    imgs = _images(golden_src, 3).cuda()
    a = model.encoder(imgs)
    b = model.encoder(imgs[1:2])
    assert torch.equal(a[1:2], b)


def test_encoder_fused_mlp_matches_the_two_launch_path(model, golden_src):
    """Option ``mlp_fused`` (default 1: fc1 + GELU + fc2 + residual of Swin stages 1 / 2 in one kernel, the hidden
    tile never in HBM) against the same encoder with fc1 and fc2 as two GEMM launches: same rounding points, so the
    features agree to fp32 summation-order noise; both stay inside the tolerance against the reference's golden."""
    imgs = _images(golden_src).cuda()
    fused = model.encoder(imgs).clone()
    model.set_option("mlp_fused", 0)
    try:
        plain = model.encoder(imgs).clone()
    finally:
        model.set_option("mlp_fused", 1)
    assert (fused - plain).abs().max().item() < 5e-3      # fp32 summation order, amplified by the fp16 roundings downstream
    for f in (fused, plain):
        assert np.abs(f.cpu().numpy() - golden_src["features"]).max() < FEAT_TOL
    big = imgs.repeat(9, 1, 1, 1)[:33]                        # > 32 images: eager launches, ragged last tile at stage 2
    assert torch.equal(model.encoder(big)[:4], model.encoder(big)[:4])
    assert (model.encoder(big)[:4] - fused).abs().max().item() < 5e-3


def test_encoder_stage_by_stage(model, dsd, cfg, golden_src):
    """Localises an encoder error: every Swin stage of the engine, rebuilt from its exported kernels (patch embed,
    LayerNorm, qkv / proj / MLP GEMMs, window attention, patch merging), against the oracle's stage outputs; the
    rebuilt schedule gives the bits of model.encoder, whose features are within tolerance for every image."""
    from oracle import ref_model as R
    from test_encoder_batch_gpu import assert_stages_close, swin_stages
    imgs = _images(golden_src, 2).cuda()
    got, feats = swin_stages(imgs, dsd)
    with torch.no_grad():
        want = R.encoder_stages(imgs, dsd)                 # list of [B,H,W,C] after patch-embed and each stage / merge
    assert_stages_close(got, want)
    assert torch.equal(feats, model.encoder(imgs))
    ref = R.encoder_forward(imgs, dsd)
    per_image = (feats - ref).abs().amax(dim=(1, 2))
    assert (per_image < FEAT_TOL).all(), per_image.tolist()


def test_decoder_against_reference_golden(model, golden_src):
    feats = torch.from_numpy(golden_src["features"][:2]).cuda()
    tgt = torch.from_numpy(golden_src["tgt"]).cuda()
    logits = model.decoder(feats, tgt)
    assert logits.shape == (2, 6, 5075)
    err = np.abs(logits.cpu().numpy() - golden_src["logits"]).max()
    print("decoder max-abs logit error vs reference:", err)
    assert err < LOGIT_TOL
    ref = torch.from_numpy(golden_src["logits"])
    top2 = ref.topk(2, -1).values
    clear = (top2[..., 0] - top2[..., 1]) > 2 * LOGIT_TOL          # positions whose winner the tolerance cannot flip
    agree = logits.argmax(-1).cpu() == ref.argmax(-1)
    print("teacher-forced argmax agreement:", agree.float().mean().item(), "clear positions:", int(clear.sum()))
    assert bool(agree[clear].all())


def test_forward_both_flavours(model, dsd, cfg, golden_src):
    from oracle import ref_model as R
    imgs = _images(golden_src, 2).cuda()
    tgt = torch.from_numpy(golden_src["tgt"]).cuda()
    out = model(imgs, tgt)                                              # app flavour
    ref = R.model_forward(imgs, tgt, dsd, cfg, drop_last=False)
    assert out.shape == ref.shape and (out - ref).abs().max().item() < 2 * LOGIT_TOL
    model.drop_last_caption = True                                      # training flavour (src/model_swin.py:100)
    try:
        out2 = model(imgs, tgt)
    finally:
        model.drop_last_caption = False
    assert out2.shape == (2, 5, 5075)
    assert (out2 - out[:, :5]).abs().max().item() < 1e-3                # causal: prefix logits unchanged


def _first_divergence(a, b):
    n = min(a.shape[1], b.shape[1])
    for r in range(a.shape[0]):
        d = np.nonzero(a[r, :n] != b[r, :n])[0]
        yield r, (int(d[0]) if d.size else None)


def test_greedy_generate_against_reference_golden(model, golden_src):
    """Tokens of /root/reference/src/inference.py::predict (fixture made by the unmodified reference)."""
    imgs = _images(golden_src).cuda()
    tokens, steps, logp = model.generate(imgs, return_logprobs=True)
    ref = golden_src["greedy_ys"]
    assert steps == ref.shape[1] - 1 and tokens.shape == ref.shape
    got = tokens.cpu().numpy()
    margin = golden_src["greedy_margin"]
    for r, c in _first_divergence(got, ref):
        if c is None:
            continue
        m = float(margin[r, c - 1])
        print(f"row {r}: first divergence at column {c}, reference top1-top2 margin {m:.4f}")
        assert m < 2 * LOGIT_TOL, "divergence at a step that is not a near-tie"
    same = sum(1 for _, c in _first_divergence(got, ref) if c is None)
    print(f"identical sequences: {same}/4")
    assert logp.shape == (4, steps) and (logp <= 0).all()


def test_generate_early_exit_and_padding(model, cfg, golden_src):
    """Rows 1-2 of the fixture both emit eos at step 19: ys has 20 columns (src/inference.py:23-25)."""
    feats = torch.from_numpy(golden_src["features"][1:3]).cuda()
    tokens, steps, _ = model.generate(encoder_out=feats)
    ref = golden_src["greedy_ys"][1:3, :20]
    got = tokens.cpu().numpy()
    # early exit: the loop stops right after the step at which the LAST row emitted its first eos (src/inference.py:23-25)
    first_eos = [int(np.nonzero(got[r, 1:] == cfg.eos)[0][0]) + 1 for r in range(2)]
    assert steps == max(first_eos) and tokens.shape == (2, steps + 1)
    if not np.array_equal(got[:, :20], ref[:, : got.shape[1]]):       # only a near-tie may move a row off the golden path
        for r, c in _first_divergence(got, ref):
            assert c is None or float(golden_src["greedy_margin"][1 + r, c - 1]) < 2 * LOGIT_TOL
    else:
        assert steps == 19 and tokens.shape == (2, 20)
    # ... and the KERNEL stops there too: it leaves its step loop on the device at most two steps after the last
    # eos (one step for the flag to reach the cluster's rank 0, one for the cluster to act on it), it does not run
    # its 16-step launch - and the launch the host had already queued behind it - to the end
    torch.cuda.synchronize()
    assert steps <= model.last_decode_steps() <= steps + 2, (steps, model.last_decode_steps())
    # max_len shorter than the sequences: length-terminated
    tokens, steps, _ = model.generate(encoder_out=feats, max_len=5)
    assert steps == 5 and tokens.shape == (2, 6) and (tokens[:, 0] == cfg.sos).all()
    torch.cuda.synchronize()
    assert model.last_decode_steps() == 5


def test_kernel_stops_on_the_device_across_clusters(model, cfg, golden_src):
    """Six clusters in one wave, rows that finish at different steps (the two golden rows that end at step 19,
    repeated): every cluster - also those whose own rows finished long before - runs exactly until the step count the
    reference's loop would reach, give or take the two steps the flag needs to travel, in ONE launch."""
    feats = torch.from_numpy(golden_src["features"]).cuda()
    feats = feats[[1, 2] * 23][:45].contiguous()                      # 45 rows = 5 full clusters + one of 5 rows
    tokens, steps, _ = model.generate(encoder_out=feats, max_len=150)
    torch.cuda.synchronize()
    one, s1, _ = model.generate(encoder_out=feats[:2], max_len=150)
    assert steps == s1 and torch.equal(tokens[:2], one)
    assert torch.equal(tokens[::2], tokens[:1].expand(23, -1)) and torch.equal(tokens[1::2], tokens[1:2].expand(22, -1))
    model.generate(encoder_out=feats, max_len=150)
    torch.cuda.synchronize()
    assert steps <= model.last_decode_steps() <= steps + 2


def test_generate_is_batch_invariant(model, golden_src):
    imgs = _images(golden_src, 4).cuda()
    all_tok, steps, _ = model.generate(imgs, max_len=40)
    for i in range(4):
        one, s1, _ = model.generate(imgs[i:i + 1], max_len=40)
        n = min(one.shape[1], all_tok.shape[1])
        row = all_tok[i, :n]
        # a single row stops at its own eos; the batch continues until all rows are done
        assert torch.equal(one[0, :n], row)


def test_incremental_decode_matches_teacher_forced(model, golden_src):
    """KV-cached step logits == full-prefix logits (same engine, both paths): argmax chain check."""
    feats = torch.from_numpy(golden_src["features"][:2]).cuda()
    tokens, steps, logp = model.generate(encoder_out=feats, max_len=12, return_logprobs=True)
    logits = model.decoder(feats, tokens[:, :-1])
    lsm = torch.log_softmax(logits, -1)
    chosen = lsm.gather(-1, tokens[:, 1:].unsqueeze(-1)).squeeze(-1)
    assert (chosen - logp).abs().max().item() < 1.5e-2
    near = (lsm.max(-1).values - chosen)       # 0 where the cached path picked the teacher-forced argmax
    assert (near < 1.5e-2).all()


@pytest.mark.parametrize("steps_per_launch", [1, 7, 64])
def test_persistent_kernel_launch_chunking(model, golden_src, steps_per_launch):
    """Splitting the step range over several launches must not change a single token."""
    feats = torch.from_numpy(golden_src["features"]).cuda()
    ref_tok, ref_steps, _ = model.generate(encoder_out=feats, max_len=40)
    model.set_option("steps_per_launch", steps_per_launch)
    try:
        tok, steps, _ = model.generate(encoder_out=feats, max_len=40)
    finally:
        model.set_option("steps_per_launch", 0)          # back to the automatic policy
    assert steps == ref_steps and torch.equal(tok, ref_tok)


def test_removed_step_graph_switch_is_an_unknown_option(model):
    """The persistent kernel is the only greedy decoder: the old step-graph switch is refused by name."""
    with pytest.raises(RuntimeError, match="unknown option"):
        model.set_option("decode_impl", 1)


@pytest.mark.parametrize("B", [1, 15, 17, 33])
def test_ragged_batches(model, golden_src, B):
    """Row counts that do not fill a 16-row cluster / 128-row GEMM tile."""
    from oracle.synth import synth_images
    imgs = synth_images(4, int(golden_src["images_seed"])).cuda()
    imgs = imgs.repeat((B + 3) // 4, 1, 1, 1)[:B].contiguous()
    tok, steps, _ = model.generate(imgs, max_len=24)
    base, _, _ = model.generate(imgs[:4] if B >= 4 else imgs, max_len=24)
    for r in range(B):
        assert torch.equal(tok[r, : base.shape[1]][: tok.shape[1]], base[r % 4 if B >= 4 else r, : tok.shape[1]])


def test_errors_are_loud(model):
    with pytest.raises(ValueError):
        model.encoder(torch.zeros(1, 3, 96, 320))
    with pytest.raises(ValueError):
        model.decoder(torch.zeros(1, 30, 256), torch.zeros(1, 151, dtype=torch.long))
    with pytest.raises(IndexError):
        model.decoder(torch.zeros(1, 30, 256), torch.full((1, 2), 9999, dtype=torch.long))
    with pytest.raises(RuntimeError):
        model.generate(torch.zeros(1, 1, 96, 320), max_len=151)
    from handwritten_math_ocr_api_b200 import FormulaRecognitionModel
    fresh = FormulaRecognitionModel(64)
    with pytest.raises(RuntimeError):
        fresh.encoder(torch.zeros(1, 1, 96, 320))
    with pytest.raises(RuntimeError):
        fresh.load_state_dict({"encoder.features.0.0.weight": torch.zeros(96, 1, 4, 4)})


def _check_tokens_against_logits(got, ys, logits, what):
    """Tokens identical, or the first divergence sits at a near-tie of the oracle's logits."""
    top2 = logits.topk(2, -1).values
    margin = (top2[..., 0] - top2[..., 1]).numpy()
    same = 0
    for r, c in _first_divergence(got, ys.numpy()):
        if c is None:
            same += 1
            continue
        m = float(margin[r, c - 1])
        assert m < DECODE_TIE_MARGIN, f"{what}: row {r} diverges at column {c} where the oracle margin is {m:.3f}"
    return same


def test_long_sequences_max_seq_len_256(golden_src):
    """BASELINE.json config 5 (T = 256): legal only when config.max_seq_len is raised before the model is built
    (SURVEY.md D6).  Exercises the 8-block (256-key) variant of the decode kernel."""
    from handwritten_math_ocr_api_b200 import FormulaRecognitionModel
    from handwritten_math_ocr_api_b200.config import Config
    from oracle import decode as odec
    from oracle.arch import ModelConfig
    from oracle.synth import synth_images, synth_state_dict

    class Config256(Config):
        max_seq_len = 256

    cfg = ModelConfig(max_seq_len=256)
    sd = synth_state_dict(cfg, seed=0, eos_bias_sigma=0.0)
    m = FormulaRecognitionModel(cfg.vocab_size, config=Config256())
    m.load_state_dict(sd)
    imgs = synth_images(3, int(golden_src["images_seed"]))
    enc = m.encoder(imgs.cuda())
    tokens, steps, _ = m.generate(encoder_out=enc, max_len=256)
    assert steps == 256 and tokens.shape == (3, 257)
    ys, lg = odec.greedy_cached(enc.cpu(), sd, cfg, max_len=256, return_logits=True)
    _check_tokens_against_logits(tokens.cpu().numpy(), ys, lg, "T=256")
    with pytest.raises(RuntimeError):
        m.generate(encoder_out=enc, max_len=257)


def test_batch_larger_than_one_wave(model, golden_src):
    """More rows than 8 x (co-resident clusters): the clusters of one launch run in several waves."""
    from oracle.synth import synth_images
    imgs = synth_images(4, int(golden_src["images_seed"])).cuda()
    base, _, _ = model.generate(imgs, max_len=20)
    B = 300
    big = imgs.repeat(B // 4, 1, 1, 1).contiguous()
    tok, steps, _ = model.generate(big, max_len=20)
    n = min(tok.shape[1], base.shape[1])
    for r in range(B):
        assert torch.equal(tok[r, :n], base[r % 4, :n])


def test_greedy_agreement_on_a_larger_sample(model, sd, cfg):
    """north_star: greedy sequences identical on >= 99.9 % of inputs, any divergence traced to a near-tie.
    64 fresh images, 60 free-running steps, against the fp32 oracle run on the SAME encoder features.  With the
    synthetic (random) checkpoint the logits are nearly flat - the oracle's own top-1/top-2 margin is below
    3e-2 on ~17 % of steps (SURVEY.md 7.2) - so what is asserted is the part that does not depend on the
    weights: EVERY divergence starts at a near-tie, and the winner's log-probability matches the oracle's
    until then."""
    from oracle import decode as odec
    from oracle.synth import synth_images
    imgs = synth_images(64, seed=4321)
    enc = model.encoder(imgs.cuda())
    tokens, steps, logp = model.generate(encoder_out=enc, max_len=60, return_logprobs=True)
    ys, lg = odec.greedy_cached(enc.cpu(), sd, cfg, max_len=60, return_logits=True)
    got = tokens.cpu().numpy()
    same = _check_tokens_against_logits(got, ys, lg, "agreement")
    ref_lp = torch.log_softmax(lg, -1).gather(-1, ys[:, 1:].unsqueeze(-1)).squeeze(-1).numpy()
    ours = logp.cpu().numpy()
    top2 = lg.topk(2, -1).values
    margin = (top2[..., 0] - top2[..., 1]).numpy()
    err, agree_steps, total, div_margins = 0.0, 0, 0, []
    for r, c in _first_divergence(got, ys.numpy()):
        n = (c - 1) if c is not None else min(ours.shape[1], ref_lp.shape[1])
        if c is not None:
            div_margins.append(float(margin[r, c - 1]))
        if n > 0:
            err = max(err, float(np.abs(ours[r, :n] - ref_lp[r, :n]).max()))
        agree_steps += n
        total += min(ours.shape[1], ref_lp.shape[1])
    print(f"identical greedy sequences: {same}/64; steps before the first divergence: {agree_steps}/{total}; "
          f"max |log p(winner) - oracle| on agreeing prefixes: {err:.4f}; oracle margins at the divergences: "
          f"max {max(div_margins) if div_margins else 0:.4f}, median {float(np.median(div_margins)) if div_margins else 0:.4f}")
    assert err < DECODE_LOGP_TOL
    assert same >= 48


# ---- beam search (not in the reference: SURVEY.md D2; definition + oracle in oracle/decode.py::beam_search) -------
def _oracle_sequence_score(enc, tokens, sd, cfg):
    """Sum of the oracle's log-softmax over the emitted tokens of each row, up to and including the first eos."""
    from oracle.ref_model import decoder_forward
    with torch.no_grad():
        lsm = torch.log_softmax(decoder_forward(enc, tokens[:, :-1], sd, cfg).float(), -1)
    out = []
    for r in range(tokens.shape[0]):
        s = 0.0
        for t in range(1, tokens.shape[1]):
            tk = int(tokens[r, t])
            s += float(lsm[r, t - 1, tk])
            if tk == cfg.eos:
                break
        out.append(s)
    return torch.tensor(out)


@pytest.mark.parametrize("beam", [2, 3, 5])
def test_beam_search_against_the_oracle(model, sd, cfg, golden_src, beam):
    from oracle import decode as odec
    feats = torch.from_numpy(golden_src["features"][:3]).cuda()
    tokens, steps, _, score = model.generate(encoder_out=feats, beam_size=beam, max_len=40)
    assert tokens.shape == (3, steps + 1) and score.shape == (3,)
    enc = feats.cpu()
    o_tok, o_score, _, _ = odec.beam_search(enc, sd, cfg, beam=beam, max_len=40)
    # (1) the score we report is the oracle's log-probability of the sequence we return (scoring + back-track)
    mine = _oracle_sequence_score(enc, tokens.cpu(), sd, cfg)
    assert (mine - score.cpu()).abs().max().item() < 3e-2
    # (2) same search result as the oracle: identical best score up to near-tie path changes
    print("beam", beam, "scores", score.cpu().tolist(), "oracle", o_score.tolist())
    assert (score.cpu() - o_score).abs().max().item() < 5e-2
    same = sum(int(tokens[r, : o_tok.shape[1]].cpu().tolist() == o_tok[r, : tokens.shape[1]].tolist()) for r in range(3))
    print("identical best hypotheses:", same, "/ 3")
    # (3) a wider beam never returns a worse hypothesis than greedy (beam search invariant on these inputs)
    g_tok, _, _ = model.generate(encoder_out=feats, max_len=40)
    greedy = _oracle_sequence_score(enc, g_tok.cpu(), sd, cfg)
    assert (score.cpu() >= greedy - 3e-2).all()


def test_beam_search_is_batch_invariant(model, golden_src):
    feats = torch.from_numpy(golden_src["features"]).cuda()
    all_tok, steps, _, all_score = model.generate(encoder_out=feats, beam_size=5, max_len=30)
    for i in range(feats.shape[0]):
        one, s1, _, sc = model.generate(encoder_out=feats[i:i + 1], beam_size=5, max_len=30)
        n = min(one.shape[1], all_tok.shape[1])
        assert torch.equal(one[0, :n], all_tok[i, :n]) and abs(float(sc[0]) - float(all_score[i])) < 1e-5


@pytest.mark.parametrize("beam", [1, 5])
def test_decode_is_bitwise_repeatable(model, beam):
    """The exchanges between the 8 CTAs of a cluster are hand-rolled (st.async + mbarrier, shared slots, named
    barriers): a race would show up as run-to-run differences.  Every cluster computes the same thing on every
    run, so tokens AND log-probabilities / scores must be bit-identical across repetitions, for a batch that mixes
    full and partial clusters and co-resident CTAs."""
    from oracle.synth import synth_images
    imgs = synth_images(8, seed=99).cuda().repeat(6, 1, 1, 1)[:45].contiguous()
    feats = model.encoder(imgs)
    ref = None
    for _ in range(6):
        out = model.generate(encoder_out=feats, max_len=70, beam_size=beam, return_logprobs=(beam == 1))
        cur = (out[0].clone(), out[2].clone() if beam == 1 else out[3].clone())
        if ref is None:
            ref = cur
        else:
            # (this test found a real one: an L2 prefetch of cache lines that another warp rewrites a step later made
            # 0.3 % of the beam-5 scores drift by up to 2e-2 - DESIGN.md 4.5)
            assert torch.equal(cur[0], ref[0]) and torch.equal(cur[1], ref[1])


def test_device_preprocessing_is_bit_identical_to_the_reference_transform(model):
    """ToTensor + Normalize(0.5, 0.5) (app/src/preprocess.py:7-12) on uint8 images, on the device."""
    from handwritten_math_ocr_api_b200.preprocess import preprocess_u8
    from handwritten_math_ocr_api_b200.synthetic import synth_images, synth_images_u8
    from torchvision import transforms
    u8 = synth_images_u8(3, seed=1234)
    u8[0, :2, :256] = torch.arange(256, dtype=torch.uint8)          # every byte value
    got = preprocess_u8(model, u8).cpu()
    norm = transforms.Normalize(mean=[0.5], std=[0.5])
    ref = torch.stack([norm(transforms.functional.to_tensor(img.numpy()[:, :, None])) for img in u8])
    assert got.shape == ref.shape == (3, 1, 96, 320) and torch.equal(got, ref)
    assert torch.equal(synth_images(3, seed=1234)[1:], got[1:])       # = the float images the benchmark feeds


def test_device_detokeniser_matches_the_reference_rule(model, cfg):
    """hmocr_pack_tokens against the Python loop of /root/reference/src/inference.py:29-40 (ids_to_strings) on token
    matrices with eos at every kind of position, sos / pad ids in the middle, rows without eos, and ragged widths."""
    from handwritten_math_ocr_api_b200.inference import ids_to_strings, packed_to_strings
    g = torch.Generator().manual_seed(7)
    idx2char = {i: f"t{i}" for i in range(cfg.vocab_size)}
    idx2char[model.pad_id], idx2char[model.sos_id], idx2char[model.eos_id] = "<pad>", "<sos>", "<eos>"
    for B, L in [(1, 1), (3, 31), (8, 32), (5, 33), (64, 151), (7, 257)]:
        t = torch.randint(3, cfg.vocab_size, (B, L), generator=g)
        t[:, 0] = model.sos_id
        for b in range(B):
            kind = b % 5
            if kind == 0 and L > 1:
                t[b, int(torch.randint(1, L, (1,), generator=g))] = model.eos_id          # one eos somewhere
            elif kind == 1 and L > 3:
                pos = torch.randint(1, L, (3,), generator=g)
                t[b, pos[0]] = model.pad_id; t[b, pos[1]] = model.sos_id; t[b, pos[2]] = model.eos_id
            elif kind == 2:
                t[b, L - 1] = model.eos_id                                                # eos in the last column
            elif kind == 3 and L > 2:
                t[b, 1] = model.eos_id; t[b, 2:] = model.pad_id                           # empty formula
            # kind 4: no eos at all
        packed, lengths = model.pack_tokens(t.cuda())
        got = packed_to_strings(packed.cpu().tolist(), lengths.cpu().tolist(), idx2char)
        want = ids_to_strings(t.tolist(), idx2char)
        assert got == want, (B, L)
        pk, ln = packed.cpu(), lengths.cpu()
        for b in range(B):
            assert (pk[b, int(ln[b]):] == model.pad_id).all()


def test_inference_predict_strings_match_the_reference_tokens(model, cfg, golden_src):
    """inference.predict (one generate call + device detokeniser) gives the strings the reference's ys decode to."""
    from handwritten_math_ocr_api_b200 import inference
    idx2char = {i: f"t{i}" for i in range(cfg.vocab_size)}
    idx2char[model.pad_id], idx2char[model.sos_id], idx2char[model.eos_id] = "<pad>", "<sos>", "<eos>"
    vocab = {v: k for k, v in idx2char.items()}
    imgs = _images(golden_src).cuda()
    got = inference.predict(imgs, model, vocab, idx2char, "cuda")
    tokens, _, _ = model.generate(imgs)
    assert got == inference.ids_to_strings(tokens.cpu().tolist(), idx2char)
    ref = inference.ids_to_strings(golden_src["greedy_ys"].tolist(), idx2char)
    assert sum(a == b for a, b in zip(got, ref)) >= 3       # near-tie divergences are checked in the token test


def test_evaluation_harness_end_to_end(model, cfg, golden_src):
    """evaluate.evaluate_model (the runnable version of src/test_model.py): labels = the engine's own greedy output
    give accuracy 1 / CER 0; corrupting one label lowers exactly that sample."""
    from handwritten_math_ocr_api_b200.evaluate import evaluate_model
    idx2char = {i: f"t{i}" for i in range(cfg.vocab_size)}
    idx2char[model.pad_id], idx2char[model.sos_id], idx2char[model.eos_id] = "<pad>", "<sos>", "<eos>"
    vocab = {v: k for k, v in idx2char.items()}
    imgs = _images(golden_src).cuda()
    tokens, steps, _ = model.generate(imgs, max_len=24)
    caps = torch.full((4, 26), model.pad_id, dtype=torch.int64)
    lens = []
    for b in range(4):
        body = [t for t in tokens[b, 1:].tolist() if t not in (model.sos_id, model.pad_id)]
        if model.eos_id in body:
            body = body[: body.index(model.eos_id)]
        seq = [model.sos_id] + body + [model.eos_id]
        caps[b, : len(seq)] = torch.tensor(seq)
        lens.append(len(seq))
    from handwritten_math_ocr_api_b200.config import Config
    c = Config(); c.max_seq_len = 24
    rows, summary = evaluate_model(model, [(imgs[:2], caps[:2], lens[:2]), (imgs[2:], caps[2:], lens[2:])], vocab, idx2char, "cuda", config=c)
    assert summary == {"accuracy": 1.0, "avg_cer": 0.0, "total_samples": 4} and [r["image_id"] for r in rows] == [0, 1, 2, 3]
    caps2 = caps.clone(); caps2[3, 1] = 3 if caps2[3, 1] != 3 else 4
    rows, summary = evaluate_model(model, [(imgs, caps2, lens)], vocab, idx2char, "cuda", config=c)
    assert summary["accuracy"] == 0.75 and rows[3]["cer"] > 0 and all(r["cer"] == 0 for r in rows[:3])


def test_gpu_image_preprocessing_is_bit_identical_to_pil_and_torchvision(model):
    """hmocr_preprocess_image_u8 (grayscale + PIL antialiased bilinear resize + ToTensor + Normalize on the GPU)
    against the reference transform itself (app/src/preprocess.py:6-16 run with the real PIL / torchvision) and the
    numpy oracle: exact equality for up- and down-scaling, both modes, degenerate and large sizes."""
    import numpy as np
    from PIL import Image
    from handwritten_math_ocr_api_b200.preprocess import preprocess_batch_gpu, preprocess_image, preprocess_image_gpu
    from oracle.preprocess import reference_preprocess
    rng = np.random.default_rng(11)
    sizes = [(96, 320), (48, 160), (200, 800), (97, 321), (1, 1), (3, 1000), (500, 7), (640, 480), (95, 319),
             (31, 333), (1200, 1600), (64, 4000)]
    pil, want = [], []
    for h, w in sizes:
        for mode in ("L", "RGB"):
            arr = rng.integers(0, 256, (h, w) if mode == "L" else (h, w, 3), dtype=np.uint8)
            img = Image.fromarray(arr, mode=mode)
            pil.append(img)
            want.append(preprocess_image(img))
            assert np.array_equal(reference_preprocess(arr), want[-1].numpy())
    got = preprocess_batch_gpu(model, pil).cpu()
    for i, w_ in enumerate(want):
        assert torch.equal(got[i:i + 1], w_), (sizes[i // 2], i % 2, (got[i:i + 1] - w_).abs().max().item())
    rgba = Image.fromarray(rng.integers(0, 256, (50, 170, 4), dtype=np.uint8), mode="RGBA")
    assert torch.equal(preprocess_image_gpu(model, rgba).cpu(), preprocess_image(rgba.convert("RGB")))


def test_gpu_dataloader_preprocessing_is_bit_identical_to_cv2(model):
    """hmocr_preprocess_cv2_u8 against src/data_loader.py:31-35 run with the real OpenCV + torchvision."""
    import cv2
    import numpy as np
    from PIL import Image
    from torchvision import transforms
    from handwritten_math_ocr_api_b200.preprocess import preprocess_dataloader_gpu
    t = transforms.Compose([transforms.Grayscale(num_output_channels=1), transforms.Resize((96, 320)),
                            transforms.ToTensor(), transforms.Normalize(mean=[0.5], std=[0.5])])
    rng = np.random.default_rng(13)
    sizes = [(96, 320), (48, 160), (192, 640), (200, 800), (97, 321), (50, 170), (500, 1300), (33, 77), (95, 319), (1, 1),
             (2, 5), (96, 1000), (300, 320), (7, 4000), (193, 641), (24, 80), (1200, 1600)]
    arrs = [rng.integers(0, 256, s, dtype=np.uint8) for s in sizes]
    want = torch.stack([t(Image.fromarray(cv2.resize(a, (320, 96)), mode='L')) for a in arrs])
    got = preprocess_dataloader_gpu(model, arrs).cpu()
    for i in range(len(sizes)):
        assert torch.equal(got[i], want[i]), (sizes[i], (got[i] - want[i]).abs().max().item())


@pytest.mark.parametrize("batch", [1, 3, 8, 32, 64, 256, 1024, 1025])
def test_encoder_graph_replays_the_same_bits(sd, cfg, golden_src, batch):
    """generate() on up to 1024 images: call 1 runs the encoder eagerly, call 2 captures it into a CUDA graph, calls 3+
    replay it from a staging copy of the images; above 1024 images every call is eager.  Tokens and log-probs must be
    the bits of the kernel-by-kernel path (encoder_graph = 0), for changing image contents too (four overlapping
    windows of one seeded image set)."""
    from handwritten_math_ocr_api_b200 import FormulaRecognitionModel
    from handwritten_math_ocr_api_b200.synthetic import synth_images
    m = FormulaRecognitionModel(cfg.vocab_size)
    m.load_state_dict(sd)
    pool = synth_images(batch + 3, seed=500).cuda()
    sets = [pool[i:i + batch] for i in range(4)]
    m.set_option("encoder_graph", 0)
    want = [m.generate(x, max_len=24, return_logprobs=True) for x in sets]
    m.set_option("encoder_graph", 1)
    for rep in range(2):
        for x, w in zip(sets, want):
            tok, steps, lp = m.generate(x, max_len=24, return_logprobs=True)
            assert steps == w[1] and torch.equal(tok, w[0]) and torch.equal(lp, w[2])


@pytest.mark.parametrize("batch,beam", [(256, 1), (128, 1), (64, 5)])
def test_decode_is_bitwise_repeatable_with_two_ctas_per_sm(model, batch, beam):
    """The same check at full occupancy (two CTAs per SM), where timing jitter is largest: this is the configuration
    in which an early L2 access to self-attention cache lines made ~1 % of the (image, run) pairs differ in their
    log-probabilities (DESIGN.md 4.4) - the 45-image test above never saw it.  256 images x 6 repetitions caught that
    build with probability > 0.99."""
    from oracle.synth import synth_images
    imgs = synth_images(8, seed=99).cuda().repeat((batch + 7) // 8, 1, 1, 1)[:batch].contiguous()
    feats = model.encoder(imgs)
    ref = None
    for _ in range(6):
        out = model.generate(encoder_out=feats, max_len=70, beam_size=beam, return_logprobs=(beam == 1))
        cur = (out[0].clone(), out[2].clone() if beam == 1 else out[3].clone())
        if ref is None:
            ref = cur
        else:
            assert torch.equal(cur[0], ref[0]) and torch.equal(cur[1], ref[1])
