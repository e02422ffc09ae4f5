"""Mirror of ``/root/reference/app/src/im2latex.py`` (what ``POST /predict`` calls):
``predict(model, image_tensor, vocab, idx2char, device) -> (formula, confidence)``.

The reference re-runs the whole Swin encoder for every generated token and syncs 3-4 times per
step (im2latex.py:25-45); here it is one ``generate`` call that also returns the chosen token's
log-softmax, from which the confidence is rebuilt with the reference's exact bookkeeping:
sum of ``log(p + 1e-10)`` over every step INCLUDING the eos step, divided by the number of
non-eos tokens (im2latex.py:33-39,50,55).  ``predict_batch`` is the tensor-batched form of the
``/predict/batch`` Python loop (app/src/main.py:546-550).

``beam_size > 1`` decodes with beam search instead (the reference app's ``DEFAULT_BEAM_SIZE``), and
``predict_nbest`` returns every image's ranked alternatives, each with the same confidence bookkeeping.
``score_formulas`` goes the other way: it scores formulas the caller already has (a user's correction, candidates
from elsewhere) against their images with one teacher-forced ``model.score`` call.
"""
from __future__ import annotations

import math
import re
from typing import Dict, List, Tuple

import torch

from .config import config

UNABLE = r"\text{Unable to detect a formula from the image. Please verify the model.}"


def tokens_to_latex(token_ids, idx2char) -> str:
    """app/src/utils.py:17-20."""
    specials = (config.sos_token, config.eos_token, config.pad_token)
    ids = [t for t in token_ids if t in idx2char and idx2char[t] not in specials]
    return ' '.join(idx2char[t] for t in ids)


def clean_latex_output(latex_str: str) -> str:
    """app/src/utils.py:22-27."""
    latex_str = re.sub(r'\\begin\s+\{', r'\\begin{', latex_str)
    latex_str = re.sub(r'\\end\s+\{', r'\\end{', latex_str)
    latex_str = re.sub(r'\{(\s+)([a-zA-Z]+)(\s+)\}', r'{\2}', latex_str)
    latex_str = re.sub(r'\\\s+\\', r'\\\\', latex_str)
    return latex_str


def load_model(model_path: str, vocab, device="cuda"):
    """im2latex.py:7-13 un-pickles a whole reference module; wrap it into the engine."""
    from .model_swin import FormulaRecognitionModel
    ref = torch.load(model_path, map_location="cpu", weights_only=False)
    sd = ref["model_state_dict"] if isinstance(ref, dict) else ref.state_dict()
    m = FormulaRecognitionModel(len(vocab), device=device)
    m.load_state_dict(sd)
    return m


def _finish(row_tokens: List[int], row_logp: List[float], eos: int, idx2char) -> Tuple[str, float]:
    out_tokens: List[int] = []
    lp_sum = 0.0
    for tok, lp in zip(row_tokens, row_logp):
        lp_sum += math.log(math.exp(lp) + 1e-10)      # log(softmax + 1e-10), im2latex.py:37
        if tok == eos:
            break
        out_tokens.append(tok)
    if not out_tokens:
        return UNABLE, 0.0
    formula = clean_latex_output(tokens_to_latex(out_tokens, idx2char))
    return formula, float(torch.exp(torch.tensor(lp_sum / len(out_tokens))).item())


def rank_hypotheses(tokens, logprobs, scores, eos: int, idx2char) -> List[Tuple[str, float, float]]:
    """One image's hypotheses, best first (``tokens[j]`` without the sos column, ``logprobs[j]``, ``scores[j]``) ->
    ``[(formula, confidence, score), ...]``: ``_finish`` on each, and a hypothesis whose formula equals a higher-ranked
    one's is dropped, so the same formula is never listed twice."""
    out: List[Tuple[str, float, float]] = []
    seen = set()
    for t, lp, sc in zip(tokens, logprobs, scores):
        formula, conf = _finish(t, lp, eos, idx2char)
        if formula not in seen:
            seen.add(formula)
            out.append((formula, conf, float(sc)))
    return out


def predict_nbest(model, image_tensors: torch.Tensor, vocab: Dict[str, int], idx2char: Dict[int, str],
                  device: str = "cuda", beam_size: int = 3, n_best: int = 3) -> List[List[Tuple[str, float, float]]]:
    """Per image, the ranked list of distinct ``(formula, confidence, score)`` among the ``n_best`` best beam
    hypotheses (``score`` = summed log-probability; entry 0 is ``predict_batch(..., beam_size=beam_size)``)."""
    model = model.to(device)
    model.eval()
    tokens, scores, logp, _ = model.generate_nbest(image_tensors, beam_size=beam_size, n_best=n_best,
                                                   max_len=config.max_seq_len)
    toks, lps, scs = tokens[:, :, 1:].cpu().tolist(), logp.cpu().tolist(), scores.cpu().tolist()
    eos = vocab[config.eos_token]
    return [rank_hypotheses(t, l, s, eos, idx2char) for t, l, s in zip(toks, lps, scs)]


def formulas_to_ids(formulas: List[str], vocab: Dict[str, int], max_seq_len: int) -> torch.Tensor:
    """Formulas in token form (vocabulary tokens separated by spaces, what ``inference.predict`` returns) ->
    int64 ``[N, 1+T]``: sos, the token ids, eos, then pad up to the longest row (T = longest formula + 1).  An unknown
    token or a formula longer than ``max_seq_len - 1`` tokens raises ValueError."""
    sos, eos, pad = vocab[config.sos_token], vocab[config.eos_token], vocab[config.pad_token]
    rows = []
    for f in formulas:
        toks = f.split()
        unknown = [t for t in toks if t not in vocab]
        if unknown:
            raise ValueError(f"token {unknown[0]!r} of formula {f!r} is not in the vocabulary")
        if len(toks) > max_seq_len - 1:
            raise ValueError(f"formula of {len(toks)} tokens exceeds max_seq_len - 1 = {max_seq_len - 1}")
        rows.append([sos] + [vocab[t] for t in toks] + [eos])
    width = max(len(r) for r in rows)
    return torch.tensor([r + [pad] * (width - len(r)) for r in rows], dtype=torch.int64)


def score_formulas(model, image_tensors: torch.Tensor, formulas: List[str], vocab: Dict[str, int],
                   idx2char: Dict[int, str], device: str = "cuda") -> List[Tuple[float, float]]:
    """Score formula ``i`` (token form) against image ``i`` -> ``[(confidence, score), ...]``.  ``score`` is the
    summed log-probability of the formula's tokens and its eos; ``confidence`` is ``predict``'s bookkeeping of the same
    per-token log-probabilities, so for ``predict``'s own output it equals ``predict``'s confidence."""
    if len(formulas) != image_tensors.shape[0]:
        raise ValueError(f"{len(formulas)} formulas for {image_tensors.shape[0]} images")
    model = model.to(device)
    model.eval()
    ids = formulas_to_ids(formulas, vocab, model.max_seq_len)
    logp, scores = model.score(image_tensors, tokens=ids)
    eos = vocab[config.eos_token]
    toks, lps, scs = ids[:, 1:].tolist(), logp.cpu().tolist(), scores.cpu().tolist()
    return [(_finish(t, l, eos, idx2char)[1], s) for t, l, s in zip(toks, lps, scs)]


def predict_batch(model, image_tensors: torch.Tensor, vocab: Dict[str, int], idx2char: Dict[int, str],
                  device: str = "cuda", beam_size: int = 1) -> List[Tuple[str, float]]:
    if beam_size > 1:
        return [hyps[0][:2] for hyps in predict_nbest(model, image_tensors, vocab, idx2char, device, beam_size, 1)]
    model = model.to(device)
    model.eval()
    tokens, steps, logp = model.generate(image_tensors, max_len=config.max_seq_len, return_logprobs=True)
    toks, lps = tokens[:, 1:].cpu().tolist(), logp.cpu().tolist()
    eos = vocab[config.eos_token]
    return [_finish(t, l, eos, idx2char) for t, l in zip(toks, lps)]


def predict(model, image_tensor: torch.Tensor, vocab: dict, idx2char: dict, device: str = "cuda", beam_size: int = 1):
    """-> (cleaned_formula, confidence_score), im2latex.py:15-56."""
    return predict_batch(model, image_tensor, vocab, idx2char, device, beam_size)[0]
