"""Drop-in mirror of ``/root/reference/src/model_res18trans.py`` (BASELINE.json config 4) backed by ``libhmocr.so``:
ResNet-18 trunk (1-channel conv1, eval-mode BatchNorm folded) -> AdaptiveAvgPool -> Linear 512->256 -> + positional
table -> 8 x TransformerEncoderLayer -> the same 8-layer decoder as the Swin model.

Two quirks of the reference are part of its semantics (SURVEY.md D7) and are kept, not fixed:

* the encoder creates a FRESH N(0,1)-initialised ``nn.Embedding(10, d_model)`` on every forward call
  (model_res18trans.py:57-59).  ``encoder(images, pos_table=None)`` draws such a table from torch's global CPU
  generator exactly like the reference does; pass ``pos_table`` (f32 ``[10, d_model]``) to pin it.
* the TransformerEncoder is ``batch_first=True`` but is fed ``[10, B, d]`` (model_res18trans.py:39-46, 61-62): its
  self-attention runs ACROSS THE IMAGES OF THE BATCH.  An image's features depend on its batch-mates, so results
  are only defined per batch composition, the batch cannot be sharded (replicas with local batches, SURVEY.md 8e),
  and B <= 256.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib
from .layout import RES18_MEM_TOKENS
from .model_swin import DecoderTransformer, FormulaRecognitionModel as _Base, _ptr, _stream


class EncoderCNN:
    """``model.encoder`` (/root/reference/src/model_res18trans.py:13-64)."""

    def __init__(self, owner: "FormulaRecognitionModel"):
        self._m = owner

    def __call__(self, x: torch.Tensor, pos_table: Optional[torch.Tensor] = None) -> torch.Tensor:
        return self.forward(x, pos_table)

    def forward(self, x: torch.Tensor, pos_table: Optional[torch.Tensor] = None) -> torch.Tensor:
        m = self._m
        m.set_pos_table(pos_table)
        return _Base._encoder_call(m, x)


class FormulaRecognitionModel(_Base):
    ENCODER_ARCH = 1
    MEM_TOKENS = RES18_MEM_TOKENS
    DECODER_LAYERS_ATTR = ("res18trans_num_decoder_layers", "num_decoder_layers")
    ENCODER_LAYERS_ATTR = ("res18trans_num_encoder_layers",)      # src/config.py:28 (independent of the decoder depth)

    def __init__(self, vocab_size: int, config=None, device=None, **kw):
        super().__init__(vocab_size, config=config, device=device, **kw)
        self.encoder = EncoderCNN(self)
        self.decoder = DecoderTransformer(self)
        self.last_pos_table: Optional[torch.Tensor] = None

    @staticmethod
    def _counts_as_parameter(key: str) -> bool:
        return key != "decoder.tgt_mask" and not key.endswith(("running_mean", "running_var", "num_batches_tracked"))

    def set_pos_table(self, pos_table: Optional[torch.Tensor]) -> torch.Tensor:
        """``None`` -> a fresh N(0,1) table, as the reference draws on every encoder call."""
        if pos_table is None:
            pos_table = torch.nn.Embedding(self.mem_tokens, self.d_model).weight.detach()
        t = pos_table.detach().to("cpu", torch.float32).contiguous()
        if tuple(t.shape) != (self.mem_tokens, self.d_model):
            raise ValueError(f"pos_table must be [{self.mem_tokens}, {self.d_model}], got {tuple(t.shape)}")
        with torch.cuda.device(self.device):
            _lib.check(self._eng.lib.hmocr_set_pos_table(self._handle(), C.c_void_p(t.data_ptr()), t.shape[0], t.shape[1],
                                                         _stream()), "hmocr_set_pos_table")
        self.last_pos_table = t
        return t

    def forward(self, images: torch.Tensor, captions: torch.Tensor, pos_table: Optional[torch.Tensor] = None):
        feats = self.encoder(images, pos_table)
        # src/model_res18trans.py:113 drops the last caption column (training flavour); keep the flag of the base class
        return self.decoder(feats, captions[:, :-1] if self.drop_last_caption else captions)

    __call__ = forward

    @torch.no_grad()
    def generate(self, images=None, max_len=None, beam_size: int = 1, return_logprobs: bool = False, encoder_out=None,
                 pos_table: Optional[torch.Tensor] = None):
        if encoder_out is None:
            self.set_pos_table(pos_table)
        return super().generate(images, max_len=max_len, beam_size=beam_size, return_logprobs=return_logprobs,
                                encoder_out=encoder_out)

    @torch.no_grad()
    def generate_nbest(self, images=None, *, encoder_out=None, beam_size: int = 3, n_best=None, max_len=None,
                       pos_table: Optional[torch.Tensor] = None):
        if encoder_out is None:
            self.set_pos_table(pos_table)
        return super().generate_nbest(images, encoder_out=encoder_out, beam_size=beam_size, n_best=n_best,
                                      max_len=max_len)

    @torch.no_grad()
    def score(self, images=None, *, encoder_out=None, tokens, return_argmax: bool = False,
              pos_table: Optional[torch.Tensor] = None):
        if encoder_out is None:
            self.set_pos_table(pos_table)
        return super().score(images, encoder_out=encoder_out, tokens=tokens, return_argmax=return_argmax)
