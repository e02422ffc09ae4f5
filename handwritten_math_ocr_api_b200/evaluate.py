"""Evaluation harness: a working version of ``/root/reference/src/test_model.py``.

The reference script cannot run as written (it passes ``mode=`` to a ``predict`` that has no such parameter,
``src/test_model.py:69`` vs ``src/inference.py:7``, and labels every row of a batch with the image ids of the first
batch, ``:79``).  The METRICS are kept exactly as the reference computes them (``calculate_metrics``, ``:47-58``):

* ``is_correct`` - exact string match of the space-joined token sequence;
* ``cer`` - ``1 - difflib.SequenceMatcher(None, pred, truth).ratio()`` over characters (the Levenshtein value the
  function computes first is always overwritten by this one).

Ground truth of a sample = ``captions[i][1 : lengths[i] - 1]`` mapped through ``idx2char`` and joined with spaces
(``:74-75``).  Predictions come from ``inference.predict`` = ONE ``generate`` call per batch.

With ``n_best > 1`` each row also gets ``in_top_n`` (the truth is among the strings of the ``n_best`` best beam
hypotheses, one more ``generate_nbest`` call per batch) and the summary ``top_n_accuracy``.

With ``score_truth=True`` the model also scores, teacher-forced, the ground truth and its own prediction of every
sample (one ``score`` call per batch over both).  That separates the two kinds of wrong prediction: a *search error*
(the model scores the truth higher than what greedy or beam search returned, so a wider search could find it) from a
*model error* (the model prefers its wrong answer).  It also gives the standard model-quality numbers: the truth's
negative log-likelihood per token, its perplexity and the teacher-forced token accuracy.
"""
from __future__ import annotations

import math
from difflib import SequenceMatcher
from typing import Dict, Iterable, List, Optional, Tuple

import torch

from . import inference
from .config import config as _default_config


def calculate_metrics(pred: str, truth: str) -> Tuple[bool, float]:
    """``src/test_model.py:47-58``."""
    cer = 1 - SequenceMatcher(None, pred, truth).ratio()
    return pred == truth, cer


def truth_string(caption, length: int, idx2char: Dict[int, str]) -> str:
    """``src/test_model.py:74-75``: drop the leading sos and the trailing eos of the padded caption."""
    return ' '.join(idx2char[int(i)] for i in caption[1:int(length) - 1])


def summarize(rows: List[dict]) -> dict:
    """``src/test_model.py:96-100``."""
    n = len(rows)
    return {
        'accuracy': sum(r['is_correct'] for r in rows) / n if n else 0.0,
        'avg_cer': sum(r['cer'] for r in rows) / n if n else 0.0,
        'total_samples': n,
    }


def score_token_rows(truths: List[List[int]], preds: List[str], vocab, config=_default_config):
    """The rows one ``score`` call of ``evaluate_model(score_truth=True)`` takes: every truth (``captions[i][:lengths[i]]``,
    sos ... eos) followed by every prediction mapped back through ``vocab`` with sos and eos added, padded with pad
    into int64 ``[2B, 1+T]``.  A row longer than ``1 + max_seq_len`` (a prediction that never emitted eos) is cut
    there; it is then scored over all ``max_seq_len`` positions."""
    sos, eos, pad = vocab[config.sos_token], vocab[config.eos_token], vocab[config.pad_token]
    rows = [list(t) for t in truths] + [[sos] + [vocab[t] for t in p.split()] + [eos] for p in preds]
    rows = [r[: 1 + config.max_seq_len] for r in rows]
    width = max(len(r) for r in rows)
    return torch.tensor([r + [pad] * (width - len(r)) for r in rows], dtype=torch.int64)


def score_columns(tokens, scores, argmax, eos: int) -> List[dict]:
    """Per sample, from a ``score`` call over ``score_token_rows`` (``B`` truths, then ``B`` predictions; host lists):
    ``truth_score``, ``truth_tokens`` (scored positions, eos included), ``pred_score`` and ``tf_token_accuracy`` (the
    share of the truth's scored positions at which the model's own top token is the truth's token)."""
    B = len(tokens) // 2
    out = []
    for i in range(B):
        body = tokens[i][1:]
        n = body.index(eos) + 1 if eos in body else len(body)
        hits = sum(int(argmax[i][t]) == int(body[t]) for t in range(n))
        out.append({'truth_score': float(scores[i]), 'truth_tokens': n, 'pred_score': float(scores[B + i]),
                    'tf_token_accuracy': hits / n})
    return out


def summarize_scores(rows: List[dict]) -> dict:
    """Pooled over every row of ``evaluate_model(score_truth=True)``: ``truth_nll_per_token`` (minus the summed truth
    scores over the summed truth tokens), ``perplexity`` (its exp), ``search_error_rate`` and ``tf_token_accuracy``
    (over all truth tokens)."""
    n_tok = sum(r['truth_tokens'] for r in rows)
    if not rows or n_tok == 0:
        return {'truth_nll_per_token': 0.0, 'perplexity': 1.0, 'search_error_rate': 0.0, 'tf_token_accuracy': 0.0}
    nll = -sum(r['truth_score'] for r in rows) / n_tok
    return {
        'truth_nll_per_token': nll,
        'perplexity': math.exp(nll),
        'search_error_rate': sum(r['search_error'] for r in rows) / len(rows),
        'tf_token_accuracy': sum(r['tf_token_accuracy'] * r['truth_tokens'] for r in rows) / n_tok,
    }


def top_n_strings(model, images, n_best: int, beam_size: int, idx2char: Dict[int, str], config=_default_config):
    """Per image, the strings of its ``n_best`` best beam hypotheses (beam width ``max(beam_size, n_best)``)."""
    tokens, _, _, _ = model.generate_nbest(images, beam_size=max(beam_size, n_best), n_best=n_best,
                                           max_len=config.max_seq_len)
    B, n, L = tokens.shape
    flat = inference.ids_to_strings(tokens.reshape(B * n, L).tolist(), idx2char, config)
    return [flat[b * n:(b + 1) * n] for b in range(B)]


def evaluate_model(model, batches: Iterable, vocab, idx2char, device=None, use_beam: bool = False,
                   beam_size: Optional[int] = None, image_ids: Optional[Iterable] = None, config=_default_config,
                   n_best: int = 1, score_truth: bool = False):
    """``evaluate_model`` (``src/test_model.py:60-87``) over an iterable of ``(images, captions, lengths)`` batches
    (what ``data_loader.get_test_loader`` yields).  Returns ``(rows, summary)``; ``rows`` are dicts with the
    reference's columns (``image_id`` is the running sample index unless ``image_ids`` supplies one per sample).
    ``n_best > 1`` adds ``in_top_n`` to every row and ``top_n_accuracy`` to the summary.  ``score_truth`` adds
    ``truth_score``, ``truth_tokens``, ``pred_score``, ``search_error`` and ``tf_token_accuracy`` to every row and
    ``summarize_scores`` to the summary."""
    model.eval()
    ids = iter(image_ids) if image_ids is not None else None
    beam = beam_size if beam_size is not None else config.beam_size
    rows: List[dict] = []
    for images, captions, lengths in batches:
        preds = inference.predict(images, model, vocab, idx2char, device, beam_size=beam, config=config,
                                  use_beam=use_beam)
        tops = top_n_strings(model, images, n_best, beam, idx2char, config) if n_best > 1 else None
        caps = captions.tolist() if hasattr(captions, "tolist") else captions
        lens = lengths.tolist() if hasattr(lengths, "tolist") else lengths
        scored = None
        if score_truth:
            tok = score_token_rows([caps[i][:int(lens[i])] for i in range(len(preds))], preds, vocab, config)
            enc = model.encoder(images)
            _, sc, am = model.score(encoder_out=torch.cat([enc, enc]), tokens=tok, return_argmax=True)
            scored = score_columns(tok.tolist(), sc.tolist(), am.tolist(), vocab[config.eos_token])
        for i, pred in enumerate(preds):
            truth = truth_string(caps[i], lens[i], idx2char)
            correct, cer = calculate_metrics(pred, truth)
            rows.append({
                'image_id': next(ids) if ids is not None else len(rows),
                'prediction': pred,
                'ground_truth': truth,
                'is_correct': correct,
                'cer': cer,
            })
            if tops is not None:
                rows[-1]['in_top_n'] = truth in tops[i]
            if scored is not None:
                rows[-1].update(scored[i])
                rows[-1]['search_error'] = not correct and scored[i]['truth_score'] > scored[i]['pred_score']
    summary = summarize(rows)
    if score_truth:
        summary.update(summarize_scores(rows))
    if n_best > 1:
        summary['top_n_accuracy'] = sum(r['in_top_n'] for r in rows) / len(rows) if rows else 0.0
    return rows, summary
