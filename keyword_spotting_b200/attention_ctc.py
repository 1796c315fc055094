"""models/attention_ctc.py ``DeployModel`` (:215-274) on a B200 -- BASELINE config 5, the consumer of the
``positional_encoding`` op.

``AttentionDeployModel.run(['model/softmax:0'], {'model/inputX:0': pcm})`` mirrors the reference's frozen-graph
call; PCM goes through the same fused front end as the rnn_ctc model (K1, n_mel = 60) and then through
``kws_attention_forward_lens``.  The reference graph has no padding mask, so a batch of utterances of different
lengths takes their lengths (``run_mel(..., lens=)``, ``forward(..., lengths=)``): each utterance is then computed
exactly as the graph computes it alone, and its output rows past ``output_lengths(lens)`` are zero.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _lib, _tensors
from .config import Config
from .rnn_ctc import DeployModel, ModelWeights
from .utils.mel import mel_filterbank


@dataclass
class AttentionConfig:
    """The inference-relevant subset of config/attention_config.py."""
    samplerate: int = 16000
    fft_size: int = 400
    hop_size: int = 160
    fmin: float = 300.0
    fmax: float = 8000.0
    n_mel: int = 60                  # :67
    combine_frame: int = 2           # :79
    num_layers: int = 3              # :80
    feed_forward_inner_size: int = 512   # :82
    multi_head_num: int = 8          # :84
    hidden_size: int = 128           # :85
    use_relu: bool = True            # :54
    label_dict: Dict[str, int] = field(default_factory=lambda: {"ni3": 1, "hao3": 2, "le4": 3})
    label_seqs: str = "1233"

    @property
    def num_classes(self) -> int:    # :87-91
        return len(self.label_dict) + 3

    @property
    def freq_size(self) -> int:
        return self.n_mel


_LAYER_FIELDS = ("w_qkv", "b_qkv", "ln1_g", "ln1_b", "w_ff1", "b_ff1", "w_ff2", "b_ff2", "ln2_g", "ln2_b")


@dataclass
class AttentionWeights:
    """fp32 host arrays; dense kernels as [in, out] (= the [1,1,in,out] kernels of tf.layers.conv2d squeezed)."""
    mel_basis: np.ndarray = None
    w_in: np.ndarray = None
    b_in: np.ndarray = None
    w_qkv: List[np.ndarray] = field(default_factory=list)
    b_qkv: List[np.ndarray] = field(default_factory=list)
    ln1_g: List[np.ndarray] = field(default_factory=list)
    ln1_b: List[np.ndarray] = field(default_factory=list)
    w_ff1: List[np.ndarray] = field(default_factory=list)
    b_ff1: List[np.ndarray] = field(default_factory=list)
    w_ff2: List[np.ndarray] = field(default_factory=list)
    b_ff2: List[np.ndarray] = field(default_factory=list)
    ln2_g: List[np.ndarray] = field(default_factory=list)
    ln2_b: List[np.ndarray] = field(default_factory=list)
    w_out: np.ndarray = None
    b_out: np.ndarray = None

    @classmethod
    def from_object(cls, o):
        """Any object with the same attribute names (e.g. the test oracle's weights)."""
        f = lambda a: np.ascontiguousarray(a, np.float32)
        w = cls(mel_basis=f(o.mel_basis), w_in=f(o.w_in), b_in=f(o.b_in), w_out=f(o.w_out), b_out=f(o.b_out))
        for name in _LAYER_FIELDS:
            setattr(w, name, [f(a) for a in getattr(o, name)])
        return w

    @classmethod
    def random_init(cls, config: AttentionConfig, seed: int = 4321):
        """glorot-uniform dense kernels (tf.layers.conv2d default), zero biases, unit layer-norm scale."""
        rng = np.random.default_rng(seed)
        N, F, C = config.hidden_size, config.feed_forward_inner_size, config.num_classes

        def glorot(i, o):
            lim = np.sqrt(6.0 / (i + o))
            return rng.uniform(-lim, lim, (i, o)).astype(np.float32)

        w = cls(mel_basis=mel_filterbank(config.samplerate, config.fft_size, config.n_mel, config.fmin,
                                         config.fmax).T.astype(np.float32).copy())
        w.w_in, w.b_in = glorot(config.combine_frame * config.n_mel, N), np.zeros(N, np.float32)
        for _ in range(config.num_layers):
            w.w_qkv.append(glorot(N, 3 * N)); w.b_qkv.append(np.zeros(3 * N, np.float32))
            w.ln1_g.append(np.ones(N, np.float32)); w.ln1_b.append(np.zeros(N, np.float32))
            w.w_ff1.append(glorot(N, F)); w.b_ff1.append(np.zeros(F, np.float32))
            w.w_ff2.append(glorot(F, N)); w.b_ff2.append(np.zeros(N, np.float32))
            w.ln2_g.append(np.ones(N, np.float32)); w.ln2_b.append(np.zeros(N, np.float32))
        w.w_out, w.b_out = glorot(N, C), np.zeros(C, np.float32)
        return w

    def validate(self, c: AttentionConfig):
        N, F, C, K = c.hidden_size, c.feed_forward_inner_size, c.num_classes, c.combine_frame * c.n_mel
        want = {"w_in": (K, N), "b_in": (N,), "w_out": (N, C), "b_out": (C,)}
        per = {"w_qkv": (N, 3 * N), "b_qkv": (3 * N,), "ln1_g": (N,), "ln1_b": (N,), "w_ff1": (N, F), "b_ff1": (F,),
               "w_ff2": (F, N), "b_ff2": (N,), "ln2_g": (N,), "ln2_b": (N,)}
        for k, shp in want.items():
            if tuple(getattr(self, k).shape) != shp:
                raise _lib.InvalidArgumentError("%s must be %r, got %r" % (k, shp, tuple(getattr(self, k).shape)))
        for k, shp in per.items():
            arrs = getattr(self, k)
            if len(arrs) != c.num_layers or any(tuple(a.shape) != shp for a in arrs):
                raise _lib.InvalidArgumentError("%s must be %d arrays of shape %r" % (k, c.num_layers, shp))
        if tuple(self.mel_basis.shape) != (c.fft_size // 2 + 1, c.n_mel):
            raise _lib.InvalidArgumentError("mel_basis must be [%d, %d]" % (c.fft_size // 2 + 1, c.n_mel))


class AttentionDeployModel:
    MAX_ROWS_PER_CALL = 1 << 20          # B*T' rows handled by one kws_attention_forward call

    def __init__(self, config: Optional[AttentionConfig] = None, weights: Optional[AttentionWeights] = None, device=None):
        self.config = config or AttentionConfig()
        self.device = _tensors.require_cuda(device)
        self.weights = weights if weights is not None else AttentionWeights.random_init(self.config)
        self.weights.validate(self.config)
        self._lib = _lib.load()
        c = self.config
        cfg = _lib.AttentionConfig(c.n_mel, c.combine_frame, c.hidden_size, c.multi_head_num, c.num_layers,
                                   c.feed_forward_inner_size, c.num_classes, int(c.use_relu))
        w = self.weights
        self._keep = []

        def p(a):
            a = np.ascontiguousarray(a, np.float32)
            self._keep.append(a)
            return a.ctypes.data_as(ctypes.c_void_p).value

        cw = _lib.AttentionWeights()
        cw.w_in, cw.b_in, cw.w_out, cw.b_out = p(w.w_in), p(w.b_in), p(w.w_out), p(w.b_out)
        for name in _LAYER_FIELDS:
            arr = getattr(cw, name)
            for l in range(c.num_layers):
                arr[l] = p(getattr(w, name)[l])
        handle = ctypes.c_void_p()
        _lib.check(self._lib.kws_attention_create(ctypes.byref(cfg), ctypes.byref(cw), self.device.index, ctypes.byref(handle)))
        self._handle = handle
        # the shared front end (K1) needs a kws_model: framing/|rFFT|/mel only, its GRU weights are never used
        fe_cfg = Config(samplerate=c.samplerate, fft_size=c.fft_size, hop_size=c.hop_size, fmin=c.fmin, fmax=c.fmax, n_mel=c.n_mel)
        fw = ModelWeights.random_init(fe_cfg, seed=0)
        fw.mel_basis = np.ascontiguousarray(w.mel_basis, np.float32)
        self._frontend = DeployModel(fe_cfg, fw, device=self.device)

    def close(self):
        if getattr(self, "_handle", None):
            self._lib.kws_attention_destroy(self._handle)
            self._handle = None
        if getattr(self, "_frontend", None):
            self._frontend.close()
            self._frontend = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def frames(self, T: int) -> int:
        return int(self._lib.kws_attention_frames(self._handle, int(T)))

    def frame_counts(self, lengths):
        """Mel frames of rows of ``lengths`` PCM samples (``DeployModel.frame_counts``), in the container type of
        ``lengths``; ``output_lengths(frame_counts(lengths))`` are the decoder's ``lens`` for ``forward(lengths=)``."""
        return self._frontend.frame_counts(lengths)

    def output_lengths(self, lens):
        """T'_b of utterances of ``lens`` valid mel frames, in the container type of ``lens`` (int, list, tuple, numpy
        or torch): the ``lens`` to give ``prediction.decode_batch`` / ``kws_ctc_decode`` for the posteriors of
        ``run_mel(mel, lens=lens)``."""
        c = self.config.combine_frame
        rule = (lambda t: t // c + 1) if c > 1 else (lambda t: t)       # kws_attention_frames
        if isinstance(lens, (torch.Tensor, np.ndarray)):
            return rule(lens)
        if isinstance(lens, (list, tuple)):
            return type(lens)(rule(int(t)) for t in lens)
        return rule(int(lens))

    def _check_lens(self, lens, B: int, T: int):
        """lens -> int32 CUDA [B].  Host values are validated (1 <= lens <= T); CUDA values are left to the kernels,
        which clamp them to [1, T] (reading them here would synchronise the stream)."""
        if not _tensors.is_host(lens):
            if tuple(lens.shape) != (B,) or lens.dtype.is_floating_point or lens.dtype == torch.bool:
                raise _lib.InvalidArgumentError("lens must be integers [%d], got %s %r" % (B, lens.dtype, tuple(lens.shape)))
            return _tensors.to_device(lens, torch.int32, self.device)
        a = np.asarray(lens.numpy() if isinstance(lens, torch.Tensor) else lens)
        if a.shape != (B,) or a.dtype.kind not in "iu":
            raise _lib.InvalidArgumentError("lens must be integers [%d], got %s %r" % (B, a.dtype, a.shape))
        if B and (a.min() < 1 or a.max() > T):
            raise _lib.InvalidArgumentError("lens must lie in [1, T = %d], got [%d, %d]" % (T, a.min(), a.max()))
        return _tensors.to_device(a.astype(np.int32), torch.int32, self.device)

    def run_mel(self, mel, want_logits: bool = False, lens=None):
        """mel ``[B, T, n_mel]`` (or ``[T, n_mel]``) -> softmax ``[B, T', C]`` [, logits].

        ``lens [B]`` (host or CUDA integers): valid mel frames per utterance, in the first rows of ``mel``.  Utterance
        b is computed exactly as a call on ``mel[b, :lens[b]]`` alone computes it, bit for bit; frames past lens[b] are
        never read and its output rows from ``output_lengths(lens)[b]`` on are zero.  Host lens must lie in [1, T]."""
        host = _tensors.is_host(mel)
        x = _tensors.to_device(mel, torch.float32, self.device)
        if x.dim() == 2:
            x = x.unsqueeze(0)
        if x.dim() != 3 or x.shape[2] != self.config.n_mel or x.shape[1] < 1:
            raise _lib.InvalidArgumentError("mel must be [B, T>=1, %d]" % self.config.n_mel)
        B, T, _ = x.shape
        ln = None if lens is None else self._check_lens(lens, B, T)
        Tp, C = self.frames(T), self.config.num_classes
        probs = torch.empty((B, Tp, C), dtype=torch.float32, device=self.device)
        logits = torch.empty_like(probs) if want_logits else None
        step = max(1, self.MAX_ROWS_PER_CALL // Tp)
        with torch.cuda.device(self.device):
            for b0 in range(0, B, step):
                b1 = min(B, b0 + step)
                _lib.check(self._lib.kws_attention_forward_lens(
                    self._handle, _tensors.ptr(x[b0:b1]), b1 - b0, T, _tensors.ptr(None if ln is None else ln[b0:b1]),
                    _tensors.ptr(probs[b0:b1]), _tensors.ptr(logits[b0:b1]) if want_logits else None,
                    _tensors.stream_ptr(self.device)))
        outs = [probs] + ([logits] if want_logits else [])
        if host:
            torch.cuda.current_stream(self.device).synchronize()
            outs = [_tensors.to_host(o) for o in outs]
        return tuple(outs) if want_logits else outs[0]

    def forward(self, inputX, want_logits: bool = False, lengths=None):
        """PCM ``[L]`` or ``[B, L]`` (float scaled by 2^-15, or int16) -> softmax ``[B, T', C]``.

        ``lengths [B]`` (host or CUDA integers): valid samples per row.  Row b is then computed bit for bit as a call on
        ``inputX[b, :lengths[b]]`` alone, on its ``frame_counts(lengths)[b]`` mel frames (``run_mel``'s ``lens``): the
        front end (``kws_frontend_mel_lens``) reads no sample past lengths[b] and stages zeros there, as past the end of
        the row alone.  Host lengths must lie in [fft_size, L]; CUDA lengths are not read on the host (no synchronisation):
        the front end clamps them to [0, L] and the attention kernels the frame counts to [1, T]."""
        host = _tensors.is_host(inputX)
        lens = None
        if lengths is not None:
            shape = tuple(inputX.shape) if isinstance(inputX, torch.Tensor) else np.shape(inputX)
            B, L = (1, shape[0]) if len(shape) == 1 else shape[:2]
            c = self.config
            if _tensors.is_host(lengths):
                a = np.asarray(lengths.numpy() if isinstance(lengths, torch.Tensor) else lengths)
                if a.shape != (B,) or a.dtype.kind not in "iu":
                    raise _lib.InvalidArgumentError("lengths must be integers [%d], got %s %r" % (B, a.dtype, a.shape))
                if B and (a.min() < c.fft_size or a.max() > L):
                    raise _lib.InvalidArgumentError("lengths must lie in [fft_size = %d, L = %d], got [%d, %d]"
                                                    % (c.fft_size, L, a.min(), a.max()))
            lengths = self._frontend._check_lengths(lengths, B, L)            # int32 CUDA [B]
            lens = self.frame_counts(lengths)
        mel = self._frontend.frontend(inputX if not host else np.asarray(inputX), lengths=lengths)
        mel_dev = _tensors.to_device(mel, torch.float32, self.device)
        outs = self.run_mel(mel_dev, want_logits, lens=lens)
        if host:
            torch.cuda.current_stream(self.device).synchronize()
            outs = tuple(_tensors.to_host(o) for o in outs) if want_logits else _tensors.to_host(outs)
        return outs

    __call__ = forward

    def run(self, fetches: Sequence[str], feed_dict: dict):
        """``sess.run`` shim for the frozen attention graph: feeds ``model/inputX:0``, fetches ``model/softmax:0``."""
        if set(feed_dict) != {"model/inputX:0"}:
            raise _lib.InvalidArgumentError("feed_dict must contain exactly 'model/inputX:0'")
        for f in fetches:
            if f != "model/softmax:0":
                raise _lib.InvalidArgumentError("unknown fetch %r (the attention graph exposes 'model/softmax:0')" % (f,))
        sm = self.forward(feed_dict["model/inputX:0"])
        return [sm for _ in fetches]
