"""The reference's greedy decode loops restated, plus the beam-search definition (oracle side).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).

* ``greedy_batched``      /root/reference/src/inference.py:7-41  (encoder once, full-prefix decoder
                          call per step, argmax, EOS-all early exit; finished rows are NOT frozen)
* ``greedy_single``       /root/reference/src/predict.py:49-67   (B=1, drops the last token even
                          when the loop ended by length)
* ``greedy_api``          /root/reference/app/src/im2latex.py:15-56 (B=1, softmax/log(p+1e-10)
                          accumulation INCLUDING the EOS step, divided by the number of non-EOS
                          tokens; encoder re-run per step in the reference - same result)
* ``greedy_cached``       same token stream as ``greedy_batched`` through ``CachedDecoder``
* ``beam_search``         NOT in the reference (SURVEY.md D2: ``beam_size`` is an unused
                          parameter).  Definition used by this repo, pinned by invariants only:
                          standard sum-of-log-softmax beam search, no length penalty.
"""
from __future__ import annotations

import math
import re
from typing import Dict, List, Optional, Tuple

import torch

from .arch import ModelConfig
from .ref_model import SD, CachedDecoder, decoder_forward, encoder_forward


def ids_to_string(seq, idx2char: Dict[int, str], cfg: ModelConfig) -> str:
    """/root/reference/src/inference.py:29-40."""
    toks = []
    for i in seq:
        t = idx2char[int(i)]
        if t in ("<sos>", "<pad>"):
            continue
        if t == "<eos>":
            break
        toks.append(t)
    return " ".join(toks)


@torch.no_grad()
def greedy_batched(images: torch.Tensor, sd: SD, cfg: ModelConfig, max_len: Optional[int] = None,
                   enc_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """-> ys int64 [B, 1+steps]."""
    enc = encoder_forward(images, sd) if enc_out is None else enc_out
    B = enc.shape[0]
    ys = torch.full((B, 1), cfg.sos, dtype=torch.long, device=enc.device)
    finished = torch.zeros(B, dtype=torch.bool, device=enc.device)
    for _ in range(max_len or cfg.max_seq_len):
        out = decoder_forward(enc, ys, sd, cfg)
        nxt = out[:, -1, :].argmax(-1, keepdim=True)
        ys = torch.cat([ys, nxt], 1)
        finished |= nxt.squeeze(1) == cfg.eos
        if finished.all():
            break
    return ys


@torch.no_grad()
def greedy_cached(enc: torch.Tensor, sd: SD, cfg: ModelConfig, max_len: Optional[int] = None,
                  return_logits: bool = False):
    """KV-cached greedy with the same stopping rule.  -> ys [B,1+steps] (and per-step logits)."""
    B = enc.shape[0]
    dec = CachedDecoder(enc, sd, cfg)
    ys = torch.full((B, 1), cfg.sos, dtype=torch.long, device=enc.device)
    finished = torch.zeros(B, dtype=torch.bool, device=enc.device)
    logits_all = []
    for _ in range(max_len or cfg.max_seq_len):
        lg = dec.step(ys[:, -1])
        if return_logits:
            logits_all.append(lg)
        nxt = lg.argmax(-1, keepdim=True)
        ys = torch.cat([ys, nxt], 1)
        finished |= nxt.squeeze(1) == cfg.eos
        if finished.all():
            break
    if return_logits:
        return ys, torch.stack(logits_all, 1)
    return ys


@torch.no_grad()
def greedy_single(image: torch.Tensor, sd: SD, cfg: ModelConfig, max_len: int = 150) -> List[int]:
    """-> token ids ``output_seq[1:-1]`` exactly as predict.py returns them (before idx2token)."""
    enc = encoder_forward(image, sd)
    seq = [cfg.sos]
    for _ in range(max_len):
        inp = torch.tensor(seq, dtype=torch.long, device=enc.device).unsqueeze(0)
        nxt = int(decoder_forward(enc, inp, sd, cfg)[:, -1, :].argmax(-1).item())
        seq.append(nxt)
        if nxt == cfg.eos:
            break
    return seq[1:-1]


def tokens_to_latex(token_ids, idx2char) -> str:
    """/root/reference/app/src/utils.py:17-20."""
    ids = [t for t in token_ids if t in idx2char and idx2char[t] not in ("<sos>", "<eos>", "<pad>")]
    return " ".join(idx2char[t] for t in ids)


def clean_latex_output(s: str) -> str:
    """/root/reference/app/src/utils.py:22-27."""
    s = re.sub(r'\\begin\s+\{', r'\\begin{', s)
    s = re.sub(r'\\end\s+\{', r'\\end{', s)
    s = re.sub(r'\{(\s+)([a-zA-Z]+)(\s+)\}', r'{\2}', s)
    s = re.sub(r'\\\s+\\', r'\\\\', s)
    return s


UNABLE = r"\text{Unable to detect a formula from the image. Please verify the model.}"


@torch.no_grad()
def greedy_api(image: torch.Tensor, sd: SD, cfg: ModelConfig, idx2char=None) -> Tuple[List[int], float, float]:
    """-> (output_tokens, log_probs_sum, confidence) with im2latex.py's exact bookkeeping."""
    enc = encoder_forward(image, sd)           # the reference recomputes this every step (same value)
    target = torch.tensor([[cfg.sos]], dtype=torch.long, device=enc.device)
    toks: List[int] = []
    lp_sum = 0.0
    for _ in range(cfg.max_seq_len):
        logits = decoder_forward(enc, target, sd, cfg)[:, -1, :]
        probs = torch.softmax(logits, -1)
        nxt = torch.argmax(probs, -1)
        lp_sum += float(torch.log(probs + 1e-10)[0, nxt.item()].item())
        if nxt.item() == cfg.eos:
            break
        toks.append(int(nxt.item()))
        target = torch.cat([target, nxt.unsqueeze(-1)], -1)
    if not toks:
        return toks, lp_sum, 0.0
    conf = float(torch.exp(torch.tensor(lp_sum / len(toks))).item())
    return toks, lp_sum, conf


@torch.no_grad()
def beam_search(enc: torch.Tensor, sd: SD, cfg: ModelConfig, beam: int, max_len: Optional[int] = None):
    """Definition (this repo's; the reference has none):

    * per image ``beam`` hypotheses; initially hypothesis 0 = [sos] with score 0, the others -inf;
    * each step every LIVE hypothesis is expanded with ``score + log_softmax(logits)`` over the
      vocabulary; a FINISHED hypothesis (it emitted eos) contributes exactly one candidate: itself,
      score frozen, token ``pad`` appended;
    * the ``beam`` best candidates are kept, ties broken towards the lower flat index
      ``hyp * V + token`` (torch.topk order on a stable sort);
    * stop after ``max_len`` steps or when every hypothesis of every image is finished;
    * result per image = highest-score hypothesis (ties -> lowest index), no length penalty.

    Scores and log-probabilities are computed in the dtype of ``enc`` (float64 inputs give a float64 search).

    -> (tokens int64 [B, 1+steps] best hypothesis, scores [B], all_tokens [B,beam,1+steps],
        all_scores [B,beam])
    """
    B, V = enc.shape[0], cfg.vocab_size
    dev = enc.device
    max_len = max_len or cfg.max_seq_len
    dec = CachedDecoder(enc, sd, cfg)
    mem_index = torch.arange(B, device=dev).repeat_interleave(beam)
    seqs = torch.full((B, beam, 1), cfg.sos, dtype=torch.long, device=dev)
    scores = torch.full((B, beam), float("-inf"), device=dev, dtype=enc.dtype)
    scores[:, 0] = 0.0
    finished = torch.zeros(B, beam, dtype=torch.bool, device=dev)
    for _ in range(max_len):
        logits = dec.step(seqs[:, :, -1].reshape(-1), mem_index)                  # [B*beam, V]
        logp = torch.log_softmax(logits.to(enc.dtype), -1).reshape(B, beam, V)
        cand = scores.unsqueeze(-1) + logp
        # finished hypotheses: single candidate (pad) with the frozen score
        fin_row = torch.full((V,), float("-inf"), device=dev, dtype=enc.dtype)
        fin_row[cfg.pad] = 0.0
        cand = torch.where(finished.unsqueeze(-1), scores.unsqueeze(-1) + fin_row, cand)
        flat = cand.reshape(B, beam * V)
        order = torch.sort(flat, dim=-1, descending=True, stable=True).indices[:, :beam]
        new_scores = torch.gather(flat, 1, order)
        parent, tok = order // V, order % V
        seqs = torch.cat([torch.gather(seqs, 1, parent.unsqueeze(-1).expand(-1, -1, seqs.shape[-1])),
                          tok.unsqueeze(-1)], -1)
        finished = torch.gather(finished, 1, parent) | (tok == cfg.eos)
        scores = new_scores
        dec.reorder((parent + torch.arange(B, device=dev).unsqueeze(1) * beam).reshape(-1))
        if finished.all():
            break
    best = scores.argmax(-1)          # first max
    tokens = seqs[torch.arange(B, device=dev), best]
    return tokens, scores[torch.arange(B, device=dev), best], seqs, scores
