"""The float64 definition of teacher-forced scoring (``hmocr_score`` / ``model.score``), built on the oracle's
``decoder_forward`` (oracle/ref_model.py).  Computed in the dtype of its input, as ``oracle.decode.beam_search`` is.
The GPU tests of ``score`` compare against it, and tests/test_score_cpu.py pins it against a per-row loop."""
import torch

from oracle.ref_model import decoder_forward


@torch.no_grad()
def score_sequences(enc: torch.Tensor, tokens: torch.Tensor, sd, cfg):
    """``decoder_forward`` on ``tokens[:, :-1]``, then

    * ``logprob[b, t] = log_softmax(logits[b, t])[tokens[b, t+1]]`` up to and including the first eos among
      ``tokens[b, 1:]``, 0 after it (a row without eos is scored over all T positions);
    * ``score[b]`` = the sum of the row of ``logprob`` in position order;
    * ``argmax[b, t]`` = the lowest index of the largest logit, ``pad`` after the first eos.

    Everything is computed in the dtype of ``enc``.  -> (logprob [B, T], score [B], argmax int64 [B, T])
    """
    T = tokens.shape[1] - 1
    logits = decoder_forward(enc, tokens[:, :-1], sd, cfg).to(enc.dtype)
    tgt = tokens[:, 1:]
    lp = torch.log_softmax(logits, -1).gather(-1, tgt.unsqueeze(-1)).squeeze(-1)
    is_eos = tgt == cfg.eos
    last = torch.where(is_eos.any(1), is_eos.int().argmax(1), torch.full_like(tgt[:, 0], T - 1))
    keep = torch.arange(T, device=tokens.device).unsqueeze(0) <= last.unsqueeze(1)
    lp = torch.where(keep, lp, torch.zeros_like(lp))
    score = torch.zeros(tokens.shape[0], dtype=enc.dtype, device=enc.device)
    for t in range(T):
        score = score + lp[:, t]
    argmax = torch.where(keep, logits.argmax(-1), torch.full_like(tgt, cfg.pad))
    return lp, score, argmax
