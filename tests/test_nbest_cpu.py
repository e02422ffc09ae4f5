"""CPU: the host side of n-best decoding - ranking / dedup / confidence of ``im2latex.predict_nbest`` and the top-n
columns of ``evaluate.evaluate_model`` - on hand-made token and log-prob tensors (no compute call)."""
import math

import torch

IDX2CHAR = {0: "<pad>", 1: "<sos>", 2: "<eos>", 3: "x", 4: "^", 5: "{", 6: "2", 7: "}", 8: "y"}
VOCAB = {v: k for k, v in IDX2CHAR.items()}
EOS, PAD = 2, 0


def test_rank_hypotheses_keeps_order_drops_duplicates_and_reports_unable():
    from handwritten_math_ocr_api_b200.im2latex import UNABLE, _finish, rank_hypotheses
    toks = [[3, 4, 6, EOS, PAD],       # x ^ 2
            [8, EOS, PAD, PAD, PAD],   # y
            [3, 4, 6, EOS, PAD],       # x ^ 2 again: dropped
            [EOS, PAD, PAD, PAD, PAD],  # empty -> UNABLE
            [PAD, 3, 4, 6, EOS]]       # pad ids are skipped: x ^ 2 a third time
    lps = [[-0.1, -0.2, -0.3, -0.05, 0.0],
           [-0.7, -0.1, 0.0, 0.0, 0.0],
           [-0.4, -0.2, -0.3, -0.05, 0.0],
           [-2.0, 0.0, 0.0, 0.0, 0.0],
           [-0.1, -0.1, -0.1, -0.1, -0.1]]
    scores = [-0.65, -0.8, -0.95, -2.0, -0.5]
    got = rank_hypotheses(toks, lps, scores, EOS, IDX2CHAR)
    assert [g[0] for g in got] == ["x ^ 2", "y", UNABLE]
    assert [g[2] for g in got] == [-0.65, -0.8, -2.0]
    assert got[2][1] == 0.0
    for (formula, conf, _), j in zip(got, (0, 1, 3)):
        assert (formula, conf) == _finish(toks[j], lps[j], EOS, IDX2CHAR)
    # the reference's bookkeeping: mean of log(p + 1e-10) over the eos step too, divided by the non-eos count
    want = math.exp(sum(math.log(math.exp(v) + 1e-10) for v in lps[0][:4]) / 3)
    assert abs(got[0][1] - want) < 1e-6


class _FakeModel:
    """Stands in for FormulaRecognitionModel: fixed greedy tokens and fixed ranked n-best tokens."""
    sos_id, eos_id, pad_id = 1, 2, 0

    def __init__(self, greedy, nbest):
        self.greedy, self.nbest = greedy, nbest
        self.nbest_calls = []

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
                if t not in (1, PAD):
                    body.append(t)
            rows.append(body)
        L = tokens.shape[1]
        packed = torch.tensor([b + [PAD] * (L - len(b)) for b in rows], dtype=torch.int32)
        return packed, torch.tensor([len(b) for b in rows], dtype=torch.int32)

    def generate_nbest(self, images, *, encoder_out=None, beam_size=3, n_best=None, max_len=None):
        self.nbest_calls.append((beam_size, n_best))
        t = self.nbest[: images.shape[0], :n_best]
        return t, torch.zeros(t.shape[:2]), torch.zeros(t.shape[0], t.shape[1], t.shape[2] - 1), t.shape[2] - 1


def test_evaluate_model_top_n_columns():
    from handwritten_math_ocr_api_b200.evaluate import evaluate_model
    S = 1
    greedy = torch.tensor([[S, 3, EOS, PAD], [S, 8, EOS, PAD], [S, 6, EOS, PAD]])
    nbest = torch.tensor([[[S, 3, EOS, PAD], [S, 8, EOS, PAD]],          # image 0: truth "x" at rank 0
                          [[S, 3, EOS, PAD], [S, 6, 7, EOS]],            # image 1: truth "2 }" at rank 1
                          [[S, 6, EOS, PAD], [S, 8, EOS, PAD]]])         # image 2: truth "y" at rank 1
    caps = torch.tensor([[S, 3, EOS, PAD], [S, 6, 7, EOS], [S, 8, EOS, PAD]])
    lens = [3, 4, 3]
    images = torch.zeros(3, 1, 96, 320)
    m = _FakeModel(greedy, nbest)
    rows, summary = evaluate_model(m, [(images, caps, lens)], VOCAB, IDX2CHAR, n_best=2, beam_size=3)
    assert [r["prediction"] for r in rows] == ["x", "y", "2"]
    assert [r["is_correct"] for r in rows] == [True, False, False]
    assert [r["in_top_n"] for r in rows] == [True, True, True]
    assert summary["top_n_accuracy"] == 1.0 and summary["accuracy"] == 1 / 3 and summary["total_samples"] == 3
    assert m.nbest_calls == [(3, 2)]
    # n_best = 1: the reference's columns and summary only, no n-best decode
    m1 = _FakeModel(greedy, nbest)
    rows1, summary1 = evaluate_model(m1, [(images, caps, lens)], VOCAB, IDX2CHAR)
    assert set(summary1) == {"accuracy", "avg_cer", "total_samples"} and all("in_top_n" not in r for r in rows1)
    assert m1.nbest_calls == []
    # the beam is widened to n_best when it is narrower; truth outside the top n
    m2 = _FakeModel(greedy, nbest)
    rows2, summary2 = evaluate_model(m2, [(images[:2], caps[:2], lens[:2])], VOCAB, IDX2CHAR, n_best=2, beam_size=1)
    assert m2.nbest_calls == [(2, 2)]
    caps_bad = caps.clone()
    caps_bad[0, 1] = 4
    rows3, summary3 = evaluate_model(_FakeModel(greedy, nbest), [(images, caps_bad, lens)], VOCAB, IDX2CHAR, n_best=2)
    assert [r["in_top_n"] for r in rows3] == [False, True, True] and abs(summary3["top_n_accuracy"] - 2 / 3) < 1e-12
