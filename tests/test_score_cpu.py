"""CPU: the host side of teacher-forced scoring - the float64 ``score_sequences`` definition (tests/score_oracle.py),
the formula -> ids conversion of ``im2latex.score_formulas`` and the score columns of ``evaluate.evaluate_model``
(no compute call)."""
import math

import pytest
import torch

IDX2CHAR = {0: "<pad>", 1: "<sos>", 2: "<eos>", 3: "x", 4: "^", 5: "{", 6: "2", 7: "}", 8: "y"}
VOCAB = {v: k for k, v in IDX2CHAR.items()}
SOS, EOS, PAD = 1, 2, 0


def test_score_sequences_matches_a_per_row_loop():
    """The batched definition against the plain one: for each row, one decoder call per scored prefix, the last
    position's log-softmax of the next token, stopping after the first eos (float64 throughout)."""
    from handwritten_math_ocr_api_b200.synthetic import synth_state_dict
    from oracle.arch import ModelConfig
    from score_oracle import score_sequences
    from oracle.ref_model import decoder_forward

    cfg = ModelConfig(vocab_size=37, num_layers=2, max_seq_len=12)
    sd = {k: v.double() if v.is_floating_point() else v
          for k, v in synth_state_dict(cfg, seed=0).items() if k.startswith("decoder.")}
    g = torch.Generator().manual_seed(7)
    enc = torch.randn(4, 30, 256, generator=g, dtype=torch.float64)
    tokens = torch.randint(3, 37, (4, 1 + 9), generator=g)
    tokens[:, 0] = SOS
    tokens[0, 4] = EOS                 # eos inside the row, garbage after it
    tokens[1, 1] = EOS                 # eos at column 1: one scored position
    tokens[2, 9] = EOS                 # eos in the last column
    tokens[3, 3] = PAD                 # no eos at all: every position is scored
    lp, score, am = score_sequences(enc, tokens, sd, cfg)
    assert lp.dtype == torch.float64 and score.dtype == torch.float64 and am.dtype == torch.int64
    T = tokens.shape[1] - 1
    for b in range(4):
        want_lp = torch.zeros(T, dtype=torch.float64)
        want_am = torch.full((T,), PAD, dtype=torch.int64)
        for t in range(T):
            logits = decoder_forward(enc[b:b + 1], tokens[b:b + 1, : t + 1], sd, cfg)[0, -1]
            want_lp[t] = torch.log_softmax(logits, -1)[tokens[b, t + 1]]
            want_am[t] = int(logits.argmax())
            if int(tokens[b, t + 1]) == EOS:
                break
        assert torch.allclose(lp[b], want_lp, rtol=0, atol=1e-10), b
        assert torch.equal(am[b], want_am), b
        s = 0.0
        for v in want_lp.tolist():
            s += v
        assert abs(float(score[b]) - s) < 1e-10
    assert int((lp[1] != 0).sum()) == 1 and int((am[1] != PAD).sum()) == 1
    assert bool((lp[3] != 0).all())


def test_formulas_to_ids_adds_sos_eos_and_pads():
    from handwritten_math_ocr_api_b200.im2latex import formulas_to_ids
    ids = formulas_to_ids(["x ^ { 2 }", "y", ""], VOCAB, max_seq_len=150)
    assert ids.dtype == torch.int64
    assert ids.tolist() == [[SOS, 3, 4, 5, 6, 7, EOS],
                            [SOS, 8, EOS, PAD, PAD, PAD, PAD],
                            [SOS, EOS, PAD, PAD, PAD, PAD, PAD]]
    # runs of spaces separate tokens like one space
    assert formulas_to_ids(["x  ^ 2"], VOCAB, 150).tolist() == [[SOS, 3, 4, 6, EOS]]


def test_formulas_to_ids_refuses_unknown_tokens_and_long_formulas():
    from handwritten_math_ocr_api_b200.im2latex import formulas_to_ids
    with pytest.raises(ValueError, match="'z'"):
        formulas_to_ids(["x ^ z"], VOCAB, 150)
    assert formulas_to_ids(["x " * 4], VOCAB, max_seq_len=5).shape == (1, 6)      # 4 tokens + eos = 5 positions
    with pytest.raises(ValueError, match="max_seq_len"):
        formulas_to_ids(["x " * 5], VOCAB, max_seq_len=5)


class _ScoringModel:
    """Stands in for FormulaRecognitionModel: fixed greedy tokens, and a ``score`` that returns fixed tensors and
    records the rows it was asked to score."""
    sos_id, eos_id, pad_id = 1, 2, 0

    def __init__(self, greedy, scores, argmax):
        self.greedy, self.scores, self.argmax = greedy, scores, argmax
        self.score_calls = []

    def eval(self):
        return self

    def generate(self, images, max_len=None, beam_size=1):
        return self.greedy[: images.shape[0]], self.greedy.shape[1] - 1, None

    def pack_tokens(self, tokens):
        rows = []
        for r in tokens.tolist():
            body = []
            for t in r:
                if t == EOS:
                    break
                if t not in (SOS, PAD):
                    body.append(t)
            rows.append(body)
        L = tokens.shape[1]
        packed = torch.tensor([b + [PAD] * (L - len(b)) for b in rows], dtype=torch.int32)
        return packed, torch.tensor([len(b) for b in rows], dtype=torch.int32)

    def encoder(self, images):
        return torch.zeros(images.shape[0], 30, 256)

    def score(self, images=None, *, encoder_out=None, tokens, return_argmax=False):
        self.score_calls.append((images, encoder_out, tokens.clone()))
        T = tokens.shape[1] - 1
        lp = torch.zeros(tokens.shape[0], T)
        return (lp, self.scores, self.argmax[:, :T]) if return_argmax else (lp, self.scores)


def test_evaluate_model_score_columns_and_summary():
    from handwritten_math_ocr_api_b200.evaluate import evaluate_model
    greedy = torch.tensor([[SOS, 3, EOS, PAD, PAD],      # "x"      truth "x"          correct
                           [SOS, 8, EOS, PAD, PAD],      # "y"      truth "2 }"        wrong, truth scored higher
                           [SOS, 6, EOS, PAD, PAD]])     # "2"      truth "x ^ 2"      wrong, truth scored lower
    caps = torch.tensor([[SOS, 3, EOS, PAD, PAD], [SOS, 6, 7, EOS, PAD], [SOS, 3, 4, 6, EOS]])
    lens = [3, 4, 5]
    # rows 0-2: truths, rows 3-5: predictions
    scores = torch.tensor([-0.5, -1.0, -6.0, -0.5, -2.0, -1.5])
    argmax = torch.tensor([[3, 2, 0, 0],                 # truth 0: x eos           -> 2 / 2
                           [6, 2, 2, 0],                 # truth 1: 2 } eos         -> 2 / 3
                           [3, 4, 6, 2],                 # truth 2: x ^ 2 eos       -> 4 / 4
                           [3, 2, 0, 0], [8, 2, 0, 0], [6, 2, 0, 0]], dtype=torch.int32)
    images = torch.zeros(3, 1, 96, 320)
    m = _ScoringModel(greedy, scores, argmax)
    rows, summary = evaluate_model(m, [(images, caps, lens)], VOCAB, IDX2CHAR, score_truth=True)
    assert len(m.score_calls) == 1
    imgs, enc, tok = m.score_calls[0]
    assert imgs is None and enc.shape == (6, 30, 256)
    assert tok.tolist() == [[SOS, 3, EOS, PAD, PAD], [SOS, 6, 7, EOS, PAD], [SOS, 3, 4, 6, EOS],
                            [SOS, 3, EOS, PAD, PAD], [SOS, 8, EOS, PAD, PAD], [SOS, 6, EOS, PAD, PAD]]
    assert [r["is_correct"] for r in rows] == [True, False, False]
    assert [r["truth_score"] for r in rows] == [-0.5, -1.0, -6.0]
    assert [r["pred_score"] for r in rows] == [-0.5, -2.0, -1.5]
    assert [r["truth_tokens"] for r in rows] == [2, 3, 4]
    assert [r["search_error"] for r in rows] == [False, True, False]
    assert [r["tf_token_accuracy"] for r in rows] == [1.0, 2 / 3, 1.0]
    nll = 7.5 / 9
    assert abs(summary["truth_nll_per_token"] - nll) < 1e-12
    assert abs(summary["perplexity"] - math.exp(nll)) < 1e-12
    assert abs(summary["search_error_rate"] - 1 / 3) < 1e-12
    assert abs(summary["tf_token_accuracy"] - 8 / 9) < 1e-12
    assert summary["total_samples"] == 3 and abs(summary["accuracy"] - 1 / 3) < 1e-12
    # without score_truth: no score call, no score columns
    m0 = _ScoringModel(greedy, scores, argmax)
    rows0, summary0 = evaluate_model(m0, [(images, caps, lens)], VOCAB, IDX2CHAR)
    assert m0.score_calls == [] and "truth_score" not in rows0[0] and "perplexity" not in summary0


def test_score_token_rows_cuts_a_prediction_without_eos():
    from handwritten_math_ocr_api_b200.config import Config
    from handwritten_math_ocr_api_b200.evaluate import score_token_rows

    class C(Config):
        max_seq_len = 4

    tok = score_token_rows([[SOS, 3, EOS]], ["x ^ 2 y"], VOCAB, C())
    assert tok.tolist() == [[SOS, 3, EOS, PAD, PAD], [SOS, 3, 4, 6, 8]]
