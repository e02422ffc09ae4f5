"""Drop-in mirror of ``/root/reference/src/model_swin.py`` backed by ``libhmocr.so``.

Same surface as the reference nn.Module (SURVEY.md section 8b):

    model = FormulaRecognitionModel(vocab_size)         # src/model_swin.py:91-95
    model.load_state_dict(checkpoint['model_state_dict'])   # src/predict.py:28-29 (517-entry layout)
    model.eval(); model.to(device)
    enc = model.encoder(images)                          # f32 [B,1,96,320] -> f32 [B,30,256]
    logits = model.decoder(enc, tgt)                     # int64 [B,T] -> f32 [B,T,V]
    logits = model(images, captions)                     # app flavour (captions whole)

plus the one new entry point the engine exists for:

    tokens, steps, logprobs = model.generate(images, max_len=150, beam_size=1)
    tokens, scores, logprobs, steps = model.generate_nbest(images, beam_size=3)     # ranked beam hypotheses
    logprobs, scores = model.score(images, tokens=tokens)                            # teacher-forced scoring

Every tensor stays a torch CUDA tensor; torch is only the allocator / stream provider.  There is
no CPU path: ``.to('cpu')`` raises, and a missing ``libhmocr.so`` raises at construction.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Iterator, Optional, Tuple

import torch

from . import _lib
from .config import config as _default_config

IMG_H, IMG_W, MEM_TOKENS = 96, 320, 30


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class _Engine:
    """Owns the ``hmocr_engine*`` handle."""

    def __init__(self, cfg: _lib.HmocrConfig, device: torch.device):
        self.lib = _lib.load()
        self.device = device
        self.handle = C.c_void_p()
        with torch.cuda.device(device):
            _lib.check(self.lib.hmocr_create(C.byref(cfg), C.byref(self.handle)), "hmocr_create")
        self.loaded = False

    def __del__(self):
        try:
            if getattr(self, "handle", None) is not None and self.handle.value:
                self.lib.hmocr_destroy(self.handle)
                self.handle = C.c_void_p()
        except Exception:
            pass


class EncoderSwin:
    """``model.encoder`` (/root/reference/src/model_swin.py:13-46)."""

    def __init__(self, owner: "FormulaRecognitionModel"):
        self._m = owner

    def __call__(self, x: torch.Tensor) -> torch.Tensor:
        return self.forward(x)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self._m._encoder_call(x)


class DecoderTransformer:
    """``model.decoder`` (/root/reference/src/model_swin.py:49-88): teacher-forced, all T positions."""

    def __init__(self, owner: "FormulaRecognitionModel"):
        self._m = owner

    def __call__(self, encoder_out: torch.Tensor, tgt: torch.Tensor) -> torch.Tensor:
        return self.forward(encoder_out, tgt)

    def forward(self, encoder_out: torch.Tensor, tgt: torch.Tensor) -> torch.Tensor:
        m = self._m
        enc = encoder_out.to(device=m.device, dtype=torch.float32).contiguous()
        tgt = tgt.to(device=m.device, dtype=torch.int64).contiguous()
        if enc.dim() != 3 or enc.shape[1] != m.mem_tokens or enc.shape[2] != m.d_model:
            raise ValueError(f"encoder_out must be [B,{m.mem_tokens},{m.d_model}], got {tuple(enc.shape)}")
        if tgt.dim() != 2 or tgt.shape[0] != enc.shape[0]:
            raise ValueError(f"tgt must be [B,T] with B={enc.shape[0]}, got {tuple(tgt.shape)}")
        B, T = tgt.shape
        if T == 0:
            return torch.empty(B, 0, m.vocab_size, dtype=torch.float32, device=m.device)
        if T > m.max_seq_len:
            raise ValueError(f"T={T} exceeds max_seq_len={m.max_seq_len} (pos_encoder / tgt_mask size)")
        if int(tgt.min()) < 0 or int(tgt.max()) >= m.vocab_size:
            raise IndexError("index out of range in self")         # what nn.Embedding raises
        m._reserve("tf", B, T)
        out = torch.empty(B, T, m.vocab_size, dtype=torch.float32, device=m.device)
        with torch.cuda.device(m.device):
            _lib.check(m._eng.lib.hmocr_decoder_forward(m._handle(), _ptr(enc), _ptr(tgt), B, T, _ptr(out), _stream()),
                       "hmocr_decoder_forward")
        return out


class FormulaRecognitionModel:
    """Mirror of ``FormulaRecognitionModel`` (/root/reference/src/model_swin.py:91-101).

    ``drop_last_caption=False`` (default) is the app/inference flavour
    (``app/src/model_swin.py:100``: ``decoder(features, captions)``); ``True`` is the training
    flavour (``src/model_swin.py:100``: ``captions[:, :-1]``).
    """

    ENCODER_ARCH = 0          # hmocr_config.encoder_arch: 0 = Swin-T
    MEM_TOKENS = MEM_TOKENS   # memory tokens per image the encoder produces
    DECODER_LAYERS_ATTR = ("swin_num_decoder_layers", "num_decoder_layers")
    ENCODER_LAYERS_ATTR = ()  # only the ResNet-18 variant has TransformerEncoder layers

    def __init__(self, vocab_size: int, config=None, device=None, drop_last_caption: bool = False,
                 sos_id: int = 1, eos_id: int = 2, pad_id: int = 0):
        cfg = config if config is not None else _default_config
        if not torch.cuda.is_available():
            raise RuntimeError("handwritten_math_ocr_api_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.type != "cuda":
            raise RuntimeError("FormulaRecognitionModel: only CUDA devices are supported (no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device(f"cuda:{torch.cuda.current_device()}")
        self.vocab_size = int(vocab_size)
        self.d_model = int(cfg.d_model)
        self.max_seq_len = int(cfg.max_seq_len)
        self.mem_tokens = self.MEM_TOKENS
        self.num_layers = 8
        for attr in self.DECODER_LAYERS_ATTR:
            if hasattr(cfg, attr):
                self.num_layers = int(getattr(cfg, attr))
                break
        self.drop_last_caption = drop_last_caption
        self.sos_id, self.eos_id, self.pad_id = sos_id, eos_id, pad_id
        enc_layers = 0
        for attr in self.ENCODER_LAYERS_ATTR:
            if hasattr(cfg, attr):
                enc_layers = int(getattr(cfg, attr))
                break
        self.enc_num_layers = enc_layers
        c = _lib.HmocrConfig(self.vocab_size, self.d_model, int(cfg.nhead), int(cfg.dim_feedforward), self.num_layers,
                             self.max_seq_len, sos_id, eos_id, pad_id, self.ENCODER_ARCH, enc_layers)
        self._eng = _Engine(c, self.device)
        self._n_params = 0
        # scratch memory is a torch tensor handed to the engine (SURVEY.md 8b "Ownership"): see _reserve
        self._workspace: Optional[torch.Tensor] = None
        self._reserved = {"gen": (0, 0, 0), "nbest": (0, 0, 0), "tf": (0, 0), "score": (0, 0)}
        self.encoder = EncoderSwin(self)
        self.decoder = DecoderTransformer(self)
        self.training = False

    # ---- nn.Module-compatible plumbing --------------------------------------------------------
    def _handle(self):
        if not self._eng.loaded:
            raise RuntimeError("weights not loaded: call load_state_dict(...) or from_reference(...) first")
        return self._eng.handle

    def eval(self):
        self.training = False
        return self

    def train(self, mode: bool = True):
        if mode:
            raise RuntimeError("the B200 engine is inference-only (no backward pass, dropout is identity)")
        return self

    def to(self, device=None, *a, **k):
        if device is None:
            return self
        d = torch.device(device)
        if d.type != "cuda":
            raise RuntimeError("FormulaRecognitionModel.to: only CUDA devices are supported (no CPU fallback)")
        if d.index is not None and d.index != self.device.index:
            raise RuntimeError(f"engine lives on {self.device}; construct a new model for {d}")
        return self

    def cuda(self, device=None):
        return self.to("cuda" if device is None else device)

    def parameters(self) -> Iterator[torch.Tensor]:
        """Only used by the reference for a parameter count (app/src/main.py:672)."""
        yield torch.empty(self._n_params, device="meta")

    def expected_keys(self):
        """Names of the reference module's ``state_dict()`` for this configuration (layout.py)."""
        from .layout import ModelConfig, state_dict_layout, state_dict_layout_res18
        mc = ModelConfig(vocab_size=self.vocab_size, max_seq_len=self.max_seq_len, num_layers=self.num_layers)
        if self.ENCODER_ARCH == 1:
            return [name for name, _, _ in state_dict_layout_res18(mc, self.enc_num_layers)]
        return [name for name, _, _ in state_dict_layout(mc)]

    def load_state_dict(self, state_dict: Dict[str, torch.Tensor], strict: bool = True):
        """Accepts the reference's 517-entry layout (or ``{'model_state_dict': ...}``).

        ``strict=True`` (the nn.Module default the reference uses, src/predict.py:29): a key the reference module
        does not have, or a missing one, raises ``RuntimeError`` like ``nn.Module.load_state_dict``;
        ``strict=False`` reports them in the returned ``_IncompatibleKeys``.  Either way the engine itself refuses to
        finalise when an entry it needs is absent or mis-shaped."""
        if "model_state_dict" in state_dict and not any(k.startswith("encoder.") for k in state_dict):
            state_dict = state_dict["model_state_dict"]        # src/utils.py:61-71 checkpoint dict
        if self._eng.loaded:
            raise RuntimeError("weights already loaded into this engine; construct a new model to reload")
        missing, unexpected = [], []
        try:
            want = set(self.expected_keys())
            missing = sorted(want - set(state_dict))
            unexpected = sorted(set(state_dict) - want)
        except Exception:                                      # a configuration layout.py cannot describe: engine checks only
            pass
        if strict and (missing or unexpected):
            raise RuntimeError("Error(s) in loading state_dict for FormulaRecognitionModel: "
                               f"missing keys {missing[:8]}{'...' if len(missing) > 8 else ''}, "
                               f"unexpected keys {unexpected[:8]}{'...' if len(unexpected) > 8 else ''}")
        lib, h = self._eng.lib, self._eng.handle
        n_params = 0
        keep = []
        with torch.cuda.device(self.device):
            for k, v in state_dict.items():
                t = v.detach().to("cpu")
                if t.dtype == torch.int64:
                    dt = 1
                else:
                    t, dt = t.to(torch.float32), 0
                    if self._counts_as_parameter(k):
                        n_params += t.numel()
                t = t.contiguous()
                keep.append(t)
                shape = (C.c_int64 * max(1, t.dim()))(*t.shape)
                _lib.check(lib.hmocr_load_weight(h, k.encode(), C.c_void_p(t.data_ptr()), shape, t.dim(), dt),
                           f"hmocr_load_weight({k})")
            _lib.check(lib.hmocr_finalize_weights(h), "hmocr_finalize_weights")
        self._n_params = n_params
        self._eng.loaded = True
        return torch.nn.modules.module._IncompatibleKeys(missing, unexpected)

    @staticmethod
    def _counts_as_parameter(key: str) -> bool:
        # encoder.features.* aliases encoder.swin.features.* (same storage); tgt_mask is a buffer
        return not key.startswith("encoder.features.") and key != "decoder.tgt_mask"

    @classmethod
    def from_reference(cls, module, config=None, device=None, **kw) -> "FormulaRecognitionModel":
        """Build from a live reference module (the API un-pickles a whole module,
        /root/reference/app/src/im2latex.py:11)."""
        sd = module.state_dict()
        vocab = sd["decoder.fc_out.weight"].shape[0]
        m = cls(vocab, config=config, device=device, **kw)
        m.load_state_dict(sd)
        return m

    # ---- scratch memory ------------------------------------------------------------------------------
    def _reserve(self, kind: str, *shape: int) -> None:
        """Make the caller-owned workspace large enough for a call of this shape.

        ``kind='gen'``: ``(batch, max_len, beam)`` of encoder / generate calls; ``kind='nbest'``: ``(batch, max_len,
        beam)`` of generate_nbest calls; ``kind='tf'``: ``(batch, T)`` of the teacher-forced decoder.  The buffer is ONE uint8 torch tensor (torch's caching allocator, current stream) sized
        by ``hmocr_workspace_bytes`` for the largest shapes seen so far and handed over with ``hmocr_set_workspace``;
        the engine allocates nothing itself.  Growing re-places every buffer (rare: shapes only ever grow)."""
        have = self._reserved[kind]
        if all(a >= b for a, b in zip(have, shape)):
            return
        self._reserved[kind] = tuple(max(a, b) for a, b in zip(have, shape))
        lib, h = self._eng.lib, self._handle()
        n = C.c_size_t()
        with torch.cuda.device(self.device):
            # the engine keeps the per-buffer maximum over every shape asked so far: `n` covers all of them
            if kind == "gen":
                b, t, k = self._reserved["gen"]
                _lib.check(lib.hmocr_workspace_bytes(h, b, t, k, C.byref(n)), "hmocr_workspace_bytes")
            elif kind == "nbest":
                b, t, k = self._reserved["nbest"]
                _lib.check(lib.hmocr_workspace_bytes(h, b, t, -k, C.byref(n)), "hmocr_workspace_bytes")
            elif kind == "score":
                b, t = self._reserved["score"]
                _lib.check(lib.hmocr_score_workspace_bytes(h, b, t, C.byref(n)), "hmocr_score_workspace_bytes")
            else:
                b, t = self._reserved["tf"]
                _lib.check(lib.hmocr_workspace_bytes(h, b, t, 0, C.byref(n)), "hmocr_workspace_bytes")
            ws = torch.empty(n.value, dtype=torch.uint8, device=self.device)
            _lib.check(lib.hmocr_set_workspace(h, _ptr(ws), n.value, _stream()), "hmocr_set_workspace")
        self._workspace = ws                                     # the old tensor goes back to torch's allocator

    def workspace_bytes(self) -> int:
        return 0 if self._workspace is None else self._workspace.numel()

    # ---- forward ------------------------------------------------------------------------------------
    def _encoder_call(self, x: torch.Tensor) -> torch.Tensor:
        x = self._images(x)
        self._reserve("gen", x.shape[0], 1, 1)
        out = torch.empty(x.shape[0], self.mem_tokens, self.d_model, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._eng.lib.hmocr_encode(self._handle(), _ptr(x), x.shape[0], _ptr(out), _stream()), "hmocr_encode")
        return out

    def _images(self, x: torch.Tensor) -> torch.Tensor:
        x = x.to(device=self.device, dtype=torch.float32).contiguous()
        if x.dim() != 4 or tuple(x.shape[1:]) != (1, IMG_H, IMG_W):
            raise ValueError(f"images must be [B,1,{IMG_H},{IMG_W}] (config.img_h x config.img_w), got {tuple(x.shape)}")
        if x.shape[0] == 0:
            raise ValueError("empty batch")
        return x

    def _memory(self, encoder_out: torch.Tensor) -> torch.Tensor:
        """Encoder output handed back by the caller: must be ``[B, mem_tokens, d_model]`` (the kernels index it raw)."""
        x = encoder_out.to(device=self.device, dtype=torch.float32).contiguous()
        if x.dim() != 3 or x.shape[0] < 1 or tuple(x.shape[1:]) != (self.mem_tokens, self.d_model):
            raise ValueError(f"encoder_out must be [B>=1,{self.mem_tokens},{self.d_model}], got {tuple(x.shape)}")
        return x

    def forward(self, images: torch.Tensor, captions: torch.Tensor) -> torch.Tensor:
        feats = self.encoder(images)
        return self.decoder(feats, captions[:, :-1] if self.drop_last_caption else captions)

    __call__ = forward

    # ---- the fast path ---------------------------------------------------------------------------
    @torch.no_grad()
    def generate_device(self, images: Optional[torch.Tensor] = None, max_len: Optional[int] = None,
                        return_logprobs: bool = False, encoder_out: Optional[torch.Tensor] = None, beam_size: int = 1):
        """``generate`` without the host synchronisation: everything stays on the stream.

        Returns ``(tokens int64 [B, 1+max_len], steps int32 [1] (device), logprobs f32 [B, max_len] | None)``
        (``beam_size > 1``: the 4th element is the best hypothesis' score, f32 ``[B]``); columns past ``steps`` hold
        ``pad``.  Used where the result feeds another stream-ordered operation (the multi-GPU token gather, a pipelined
        device-to-host copy) so the GPU never idles waiting for the host."""
        max_len = int(max_len if max_len is not None else self.max_seq_len)
        lib = self._eng.lib
        x = self._images(images) if encoder_out is None else self._memory(encoder_out)
        B = x.shape[0]
        if not 1 <= max_len <= self.max_seq_len:
            raise RuntimeError(f"max_len={max_len} outside [1, {self.max_seq_len}] (size of pos_encoder, src/model_swin.py:54)")
        self._reserve("gen", B, max_len, int(beam_size))
        tokens = torch.empty(B, max_len + 1, dtype=torch.int64, device=self.device)
        logp = torch.empty(B, max_len, dtype=torch.float32, device=self.device) if return_logprobs else None
        steps = torch.zeros(1, dtype=torch.int32, device=self.device)
        score = torch.zeros(B, dtype=torch.float32, device=self.device) if beam_size > 1 else None
        with torch.cuda.device(self.device):
            fn = lib.hmocr_generate if encoder_out is None else lib.hmocr_generate_from_memory
            _lib.check(fn(self._handle(), _ptr(x), B, max_len, int(beam_size), _ptr(tokens), _ptr(logp), _ptr(steps),
                          _ptr(score), _stream()), "hmocr_generate")
        if beam_size > 1:
            return tokens, steps, logp, score
        return tokens, steps, logp

    @torch.no_grad()
    def generate(self, images: Optional[torch.Tensor] = None, max_len: Optional[int] = None, beam_size: int = 1,
                 return_logprobs: bool = False, encoder_out: Optional[torch.Tensor] = None):
        """Greedy (beam_size=1) or beam decode in ONE library call.

        Returns ``(tokens int64 [B, 1+steps], steps, logprobs f32 [B, steps] | None)`` where
        ``tokens`` is exactly the ``ys`` of /root/reference/src/inference.py:15-25 (column 0 = sos;
        decoding stops at the first step after which every row has emitted eos, or at max_len).
        """
        max_len = int(max_len if max_len is not None else self.max_seq_len)
        lib = self._eng.lib
        x = self._images(images) if encoder_out is None else self._memory(encoder_out)
        B = x.shape[0]
        if not 1 <= max_len <= self.max_seq_len:
            raise RuntimeError(f"max_len={max_len} outside [1, {self.max_seq_len}] (size of pos_encoder, src/model_swin.py:54)")
        self._reserve("gen", B, max_len, int(beam_size))
        tokens = torch.empty(B, max_len + 1, dtype=torch.int64, device=self.device)
        logp = torch.empty(B, max_len, dtype=torch.float32, device=self.device) if return_logprobs else None
        steps = torch.zeros(1, dtype=torch.int32, device=self.device)
        score = torch.zeros(B, dtype=torch.float32, device=self.device) if beam_size > 1 else None
        with torch.cuda.device(self.device):
            fn = lib.hmocr_generate if encoder_out is None else lib.hmocr_generate_from_memory
            _lib.check(fn(self._handle(), _ptr(x), B, max_len, int(beam_size), _ptr(tokens), _ptr(logp), _ptr(steps),
                          _ptr(score), _stream()), "hmocr_generate")
        n = int(steps.item())
        out_lp = logp[:, :n] if return_logprobs else None
        if beam_size > 1:
            return tokens[:, : n + 1], n, out_lp, score
        return tokens[:, : n + 1], n, out_lp

    @torch.no_grad()
    def generate_nbest(self, images: Optional[torch.Tensor] = None, *, encoder_out: Optional[torch.Tensor] = None,
                       beam_size: int = 3, n_best: Optional[int] = None, max_len: Optional[int] = None):
        """The ``n_best`` (default ``beam_size``) best hypotheses of a beam search per image, ranked by score.

        Returns ``(tokens int64 [B, n, 1+steps], scores f32 [B, n], logprobs f32 [B, n, steps], steps)``.  Rank 0 is
        what ``generate(beam_size=beam_size)`` returns; ``logprobs`` holds each emitted token's log-softmax (0 after the
        hypothesis' eos) and ``scores`` is its fp32 sum in step order.  ``beam_size=1`` gives the greedy sequence."""
        beam = int(beam_size)
        n = beam if n_best is None else int(n_best)
        max_len = int(max_len if max_len is not None else self.max_seq_len)
        x = self._images(images) if encoder_out is None else self._memory(encoder_out)
        B = x.shape[0]
        if not 1 <= max_len <= self.max_seq_len:
            raise RuntimeError(f"max_len={max_len} outside [1, {self.max_seq_len}] (size of pos_encoder, src/model_swin.py:54)")
        if 1 <= beam <= 5:                      # otherwise the library call below names the problem
            self._reserve("nbest", B, max_len, beam)
        tokens = torch.empty(B, max(n, 0), max_len + 1, dtype=torch.int64, device=self.device)
        logp = torch.empty(B, max(n, 0), max_len, dtype=torch.float32, device=self.device)
        scores = torch.empty(B, max(n, 0), dtype=torch.float32, device=self.device)
        steps = torch.zeros(1, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._eng.lib.hmocr_generate_nbest(self._handle(), _ptr(x), int(encoder_out is not None), B,
                                                          max_len, beam, n, _ptr(tokens), _ptr(logp), _ptr(scores),
                                                          _ptr(steps), _stream()), "hmocr_generate_nbest")
        t = int(steps.item())
        return tokens[:, :, : t + 1], scores, logp[:, :, :t], t

    @torch.no_grad()
    def score(self, images: Optional[torch.Tensor] = None, *, encoder_out: Optional[torch.Tensor] = None,
              tokens: torch.Tensor, return_argmax: bool = False):
        """Teacher-forced scoring of given sequences: how likely each formula is for its image.

        ``tokens`` int64 ``[B, 1+T]`` in the layout ``generate`` returns (column 0 = sos, then the scored tokens; what
        follows a row's first eos is ignored).  Returns ``(logprobs f32 [B, T], scores f32 [B])`` - the log-softmax of
        each scored token up to and including the row's first eos (0 after it) and its fp32 sum in position order, the
        definition of ``generate_nbest``'s scores - plus ``argmax`` int32 ``[B, T]`` (the model's own top token at each
        position, lowest index on ties, pad after eos) when ``return_argmax``.  The logits are never materialised.
        A bad shape raises ValueError, an id outside the vocabulary IndexError, T outside [1, max_seq_len]
        RuntimeError."""
        if (images is None) == (encoder_out is None):
            raise ValueError("score: pass exactly one of images and encoder_out")
        x = self._images(images) if encoder_out is None else self._memory(encoder_out)
        B = x.shape[0]
        tok = tokens.to(device=self.device, dtype=torch.int64).contiguous()
        if tok.dim() != 2 or tok.shape[0] != B or tok.shape[1] < 1:
            raise ValueError(f"tokens must be [B,1+T] with B={B}, got {tuple(tok.shape)}")
        if int(tok.min()) < 0 or int(tok.max()) >= self.vocab_size:
            raise IndexError("index out of range in self")         # what nn.Embedding raises
        T = tok.shape[1] - 1
        if 1 <= T <= self.max_seq_len:                              # otherwise the library call below names the problem
            self._reserve("score", B, T)
        logp = torch.empty(B, T, dtype=torch.float32, device=self.device)
        scores = torch.empty(B, dtype=torch.float32, device=self.device)
        argmax = torch.empty(B, T, dtype=torch.int32, device=self.device) if return_argmax else None
        with torch.cuda.device(self.device):
            _lib.check(self._eng.lib.hmocr_score(self._handle(), _ptr(x), int(encoder_out is not None), B, T, _ptr(tok),
                                                 _ptr(logp), _ptr(scores), _ptr(argmax), _stream()), "hmocr_score")
        if return_argmax:
            return logp, scores, argmax
        return logp, scores

    @torch.no_grad()
    def pack_tokens(self, tokens: torch.Tensor):
        """Detokenise on the device (the per-id Python loop of /root/reference/src/inference.py:29-40): drops sos /
        pad ids, stops at the first eos.  ``tokens`` int64 ``[B, L]`` (CUDA) -> ``(packed int32 [B, L], lengths int32
        [B])``, both on the device; row ``b`` keeps ``packed[b, :lengths[b]]``."""
        t = tokens.to(device=self.device, dtype=torch.int64).contiguous()
        B, L = t.shape
        packed = torch.empty(B, L, dtype=torch.int32, device=self.device)
        lengths = torch.empty(B, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._eng.lib.hmocr_pack_tokens(self._handle(), _ptr(t), B, L, _ptr(lengths), _ptr(packed), _stream()),
                       "hmocr_pack_tokens")
        return packed, lengths

    def set_option(self, name: str, value: int) -> None:
        """Engine options of ``hmocr_set_option`` (``decode_impl``, ``steps_per_launch``, ``encoder_graph``, ``mlp_fused``, ...:
        include/hmocr.h lists them)."""
        _lib.check(self._eng.lib.hmocr_set_option(self._eng.handle, name.encode(), int(value)), "hmocr_set_option")
        # options change which scratch buffers a call uses (step graph / tracing): plan again
        self._reserved = {"gen": (0, 0, 0), "nbest": (0, 0, 0), "tf": (0, 0), "score": (0, 0)}

    def last_decode_steps(self) -> int:
        """Decode steps the persistent kernel executed in the last ``generate`` call (after a stream synchronise): the
        kernel leaves its step loop on the device right after every row has emitted eos."""
        n = C.c_int32()
        _lib.check(self._eng.lib.hmocr_last_decode_steps(self._eng.handle, C.byref(n)), "hmocr_last_decode_steps")
        return int(n.value)

    def last_timings_ms(self) -> Tuple[float, float]:
        enc, dec = C.c_float(), C.c_float()
        _lib.check(self._eng.lib.hmocr_last_timings(self._eng.handle, C.byref(enc), C.byref(dec)), "hmocr_last_timings")
        return enc.value, dec.value
