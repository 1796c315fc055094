"""Drop-in for the deployment model of models/rnn_ctc.py (``DeployModel``, :113-166).

The reference builds a TF graph and exposes named tensors that ``detector.py``
drives through ``sess.run`` (:190-193).  Here the graph body is the CUDA path
behind ``kws_deploy_forward`` / ``kws_gru_forward``; the entry points keep the
reference's names and call conventions:

    model = DeployModel(config, weights)
    softmax, state = model.run(['model/softmax:0', 'model/rnn_states:0'],
                               feed_dict={'model/inputX:0': pcm,
                                          'model/rnn_initial_states:0': state})

``inputX`` is float32 PCM ``[L]`` exactly as in the reference, or a batch
``[S, L]`` (float32 or int16), or mel frames ``[n, M]`` / ``[S, n, M]`` through
``run_mel`` (the commented mel-input form, models/rnn_ctc.py:150-153).  State is
functional: ``[num_layers, S, hidden]`` in, same shape out.  numpy in -> numpy
out; CUDA torch tensors in -> CUDA torch tensors out.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib, _tensors
from .config import Config
from .utils.mel import mel_filterbank

INPUT_X = "model/inputX:0"                       # main.py:339-342 output/input names
INITIAL_STATES = "model/rnn_initial_states:0"
RNN_STATES = "model/rnn_states:0"
SOFTMAX = "model/softmax:0"
LOGIT = "model/logit:0"


@dataclass
class ModelWeights:
    """fp32 parameters in the TF variable layout (see include/kws_b200.h).

    TF names (SURVEY.md 8f-3): ``model/drnn/multi_rnn_cell/cell_{l}/gru_cell/
    {gates,candidate}/{kernel,bias}``, ``model/weightsClasses``, ``model/biasesClasses``.
    """
    mel_basis: np.ndarray                                   # [fft_size/2 + 1, M]
    gates_kernel: List[np.ndarray] = field(default_factory=list)   # [in+H, 2H]
    gates_bias: List[np.ndarray] = field(default_factory=list)     # [2H]
    cand_kernel: List[np.ndarray] = field(default_factory=list)    # [in+H, H]
    cand_bias: List[np.ndarray] = field(default_factory=list)      # [H]
    fc_w: Optional[np.ndarray] = None                       # [H, C]
    fc_b: Optional[np.ndarray] = None                       # [C]

    @classmethod
    def from_arrays(cls, mel_basis, gates_kernel, gates_bias, cand_kernel, cand_bias, fc_w, fc_b):
        f = lambda a: np.ascontiguousarray(a, dtype=np.float32)
        return cls(f(mel_basis), [f(a) for a in gates_kernel], [f(a) for a in gates_bias],
                   [f(a) for a in cand_kernel], [f(a) for a in cand_bias], f(fc_w), f(fc_b))

    @classmethod
    def from_frozen_graph(cls, path_or_bytes, n_mel: Optional[int] = None, fft_size: int = 400):
        """Weights of a frozen deployment ``graph.pb`` (main.py:339-348), read without TensorFlow
        (keyword_spotting_b200/graph_pb.py).  ``fft_size``: the model's frame; its mel basis is
        ``[fft_size/2 + 1, n_mel]``."""
        from . import graph_pb
        return graph_pb.rnn_ctc_weights(graph_pb.load_graph(path_or_bytes), n_mel=n_mel, fft_size=fft_size)

    @classmethod
    def random_init(cls, config: Config, seed: int = 1234):
        """Random-init weights of the reference architecture: Xavier-normal GRU
        kernels (models/rnn_ctc.py:230-232), gate bias 1 / candidate bias 0 (TF
        GRUCell), truncated-normal FC (models/rnn_ctc.py:265-273)."""
        rng = np.random.default_rng(seed)
        H, C, M = config.hidden_size, config.num_classes, config.n_mel
        w = cls(mel_basis=mel_filterbank(config.samplerate, config.fft_size, M, config.fmin,
                                         config.fmax).T.astype(np.float32).copy())
        for layer in range(config.num_layers):
            fan_in = (M if layer == 0 else H) + H
            w.gates_kernel.append((rng.standard_normal((fan_in, 2 * H)) * np.sqrt(2.0 / (fan_in + 2 * H))).astype(np.float32))
            w.gates_bias.append(np.ones(2 * H, np.float32))
            w.cand_kernel.append((rng.standard_normal((fan_in, H)) * np.sqrt(2.0 / (fan_in + H))).astype(np.float32))
            w.cand_bias.append(np.zeros(H, np.float32))
        fc = rng.standard_normal((H, C))
        bad = np.abs(fc) > 2.0
        while bad.any():
            fc[bad] = rng.standard_normal(int(bad.sum()))
            bad = np.abs(fc) > 2.0
        w.fc_w = fc.astype(np.float32)
        w.fc_b = np.zeros(C, np.float32)
        return w

    def validate(self, config: Config):
        H, C, M = config.hidden_size, config.num_classes, config.n_mel
        if self.mel_basis.shape != (config.fft_size // 2 + 1, M):
            raise _lib.InvalidArgumentError("mel_basis must be [%d, %d], got %r" % (config.fft_size // 2 + 1, M, self.mel_basis.shape))
        if not (len(self.gates_kernel) == len(self.gates_bias) == len(self.cand_kernel) == len(self.cand_bias) == config.num_layers):
            raise _lib.InvalidArgumentError("need weights for %d layers" % config.num_layers)
        for l in range(config.num_layers):
            fan_in = (M if l == 0 else H) + H
            for name, arr, shape in (("gates_kernel", self.gates_kernel[l], (fan_in, 2 * H)),
                                     ("gates_bias", self.gates_bias[l], (2 * H,)),
                                     ("cand_kernel", self.cand_kernel[l], (fan_in, H)),
                                     ("cand_bias", self.cand_bias[l], (H,))):
                if tuple(arr.shape) != shape:
                    raise _lib.InvalidArgumentError("%s[%d] must be %r, got %r" % (name, l, shape, tuple(arr.shape)))
        if tuple(self.fc_w.shape) != (H, C) or tuple(self.fc_b.shape) != (C,):
            raise _lib.InvalidArgumentError("fc_w/fc_b must be [%d,%d]/[%d]" % (H, C, C))


@dataclass
class OctbitMatrix:
    """One converted MatMul of the octbit graph: qint8 Const ``[out, in]`` + the op's ``scale`` / ``bias`` attrs
    (octbit/octbit_graph.py:191-215, 527-536)."""
    weight_q: np.ndarray
    scale: float
    bias: np.ndarray


@dataclass
class OctbitModelWeights:
    """The OctbitMatMul constants of ``graph_octbit.pb``: GRU layers by index (the rewriter converts every layer but
    cell_0, octbit/octbit_graph.py:218-225) and the FC."""
    gates: dict = field(default_factory=dict)        # layer -> OctbitMatrix [2H, in+H]
    candidate: dict = field(default_factory=dict)    # layer -> OctbitMatrix [H, in+H]
    fc: Optional[OctbitMatrix] = None                # [C, H]

    @classmethod
    def from_float(cls, weights: "ModelWeights", layers=None, fc: bool = True, device=None):
        """What the reference's GraphRewriter produces from the float graph: ``octize_weight_int8_signed`` on the
        kernels of every layer but the first (or ``layers``) and on the FC."""
        from .octbit.octbit_graph import octize_weight_int8_signed
        L = len(weights.gates_kernel)
        layers = list(range(1, L)) if layers is None else list(layers)

        def octize(w):
            wq, scale, bias = octize_weight_int8_signed(np.ascontiguousarray(w, np.float32), device=device)
            return OctbitMatrix(np.ascontiguousarray(wq, np.int8), float(np.float32(scale)), np.ascontiguousarray(bias, np.float32))

        ow = cls()
        for l in layers:
            ow.gates[l] = octize(weights.gates_kernel[l])
            ow.candidate[l] = octize(weights.cand_kernel[l])
        if fc:
            ow.fc = octize(weights.fc_w)
        return ow


class DeployModel:
    """models/rnn_ctc.py:113-166 on a B200.  Owns a ``kws_model`` handle."""

    def __init__(self, config: Optional[Config] = None, weights: Optional[ModelWeights] = None, device=None,
                 precision: str = "tc", frontend: Optional[str] = None):
        """``precision``: ``"tc"`` (default) = tcgen05 tensor cores, fp16 operands / fp32 accumulate and state;
        ``"fp32"`` = every product in fp32 on the CUDA cores (the accuracy baseline).
        ``frontend``: ``"fft"`` (default) or ``"tc"`` (hop-block DFTs on tcgen05; int16 PCM) -- same results, same speed.
        Both are 400/160 kernels: a model of any other ``fft_size`` / ``hop_size`` runs the general DFT front end
        (csrc/frontend_dft.cu) whatever ``frontend`` says."""
        self.config = config or Config()
        self.device = _tensors.require_cuda(device)
        self.weights = weights if weights is not None else ModelWeights.random_init(self.config)
        self.weights.validate(self.config)
        self._lib = _lib.load()
        cfg = _lib.ModelConfig(self.config.n_mel, self.config.hidden_size, self.config.num_layers,
                               self.config.num_classes, self.config.fft_size, self.config.hop_size)
        w = self.weights
        self._keep = [np.ascontiguousarray(a, np.float32) for a in
                      [w.mel_basis, *w.gates_kernel, *w.gates_bias, *w.cand_kernel, *w.cand_bias, w.fc_w, w.fc_b]]
        cw = _lib.ModelWeights()
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p).value
        L = self.config.num_layers
        cw.mel_basis = p(self._keep[0])
        for l in range(L):
            cw.gates_kernel[l] = p(self._keep[1 + l])
            cw.gates_bias[l] = p(self._keep[1 + L + l])
            cw.cand_kernel[l] = p(self._keep[1 + 2 * L + l])
            cw.cand_bias[l] = p(self._keep[1 + 3 * L + l])
        cw.fc_w = p(self._keep[1 + 4 * L])
        cw.fc_b = p(self._keep[2 + 4 * L])
        handle = ctypes.c_void_p()
        _lib.check(self._lib.kws_model_create(ctypes.byref(cfg), ctypes.byref(cw), self.device.index,
                                              ctypes.byref(handle)))
        self._handle = handle
        self.octbit = None
        self._keep_oct = None
        self.set_precision(precision)
        if frontend is not None:
            self.set_frontend(frontend)
        self.frontend_kind = {_lib.FRONTEND_FFT: "fft", _lib.FRONTEND_TC: "tc"}[int(self._lib.kws_model_get_frontend(self._handle))]

    def set_frontend(self, frontend: str):
        modes = {"fft": _lib.FRONTEND_FFT, "tc": _lib.FRONTEND_TC}
        if frontend not in modes:
            raise _lib.InvalidArgumentError("frontend must be 'fft' or 'tc'")
        _lib.check(self._lib.kws_model_set_frontend(self._handle, modes[frontend]))
        self.frontend_kind = frontend

    @classmethod
    def from_octbit_graph(cls, path_or_bytes, config: Optional[Config] = None, device=None, n_mel: Optional[int] = None):
        """The reference's deployable artefact ``graph_octbit.pb`` (main.py:357-371): float cell_0 + OctbitMatMul
        everywhere else, read without TensorFlow and run through the octbit kernels."""
        from . import graph_pb
        fft_size = config.fft_size if config is not None else Config.fft_size
        weights, octw = graph_pb.rnn_ctc_octbit_weights(graph_pb.load_graph(path_or_bytes), n_mel=n_mel, fft_size=fft_size)
        cfg = config or Config(n_mel=weights.mel_basis.shape[1], num_layers=len(weights.gates_kernel))
        model = cls(cfg, weights, device=device, precision="fp32")
        model.set_octbit(octw)
        return model

    def set_octbit(self, octw: Optional["OctbitModelWeights"]):
        """Switch every forward of this model to the octbit-rewritten graph (``None``: back to the float graph).
        Converted MatMuls use per-stream activation ranges, i.e. the reference's batch-1 semantics."""
        if octw is None:
            _lib.check(self._lib.kws_model_set_octbit(self._handle, None))
            self.octbit = None
            self._keep_oct = None
            return
        cw = _lib.OctbitWeights()
        keep = []

        def put(mat, rows, cols, what):
            wq = np.ascontiguousarray(mat.weight_q, np.int8)
            ob = np.ascontiguousarray(mat.bias, np.float32).reshape(-1)
            if wq.shape != (rows, cols) or ob.shape != (rows,):
                raise _lib.InvalidArgumentError("%s: weight_q must be [%d, %d] int8 and bias [%d], got %r / %r"
                                                % (what, rows, cols, rows, wq.shape, ob.shape))
            keep.extend([wq, ob])
            return wq.ctypes.data_as(ctypes.c_void_p).value, float(mat.scale), ob.ctypes.data_as(ctypes.c_void_p).value

        H, C, L = self.config.hidden_size, self.config.num_classes, self.config.num_layers
        if set(octw.gates) != set(octw.candidate):
            raise _lib.InvalidArgumentError("gates and candidate must be converted for the same layers")
        for l in octw.gates:
            if not 0 <= l < L:
                raise _lib.InvalidArgumentError("layer %r out of range" % (l,))
            K = (self.config.n_mel if l == 0 else H) + H
            cw.gates_wq[l], cw.gates_scale[l], cw.gates_obias[l] = put(octw.gates[l], 2 * H, K, "gates[%d]" % l)
            cw.cand_wq[l], cw.cand_scale[l], cw.cand_obias[l] = put(octw.candidate[l], H, K, "candidate[%d]" % l)
        if octw.fc is not None:
            cw.fc_wq, cw.fc_scale, cw.fc_obias = put(octw.fc, C, H, "fc")
        with torch.cuda.device(self.device):
            _lib.check(self._lib.kws_model_set_octbit(self._handle, ctypes.byref(cw)))
        self.octbit = octw
        self._keep_oct = keep

    def set_precision(self, precision: str):
        modes = {"tc": _lib.PRECISION_TC_FP16, "fp32": _lib.PRECISION_FP32}
        if precision not in modes:
            raise _lib.InvalidArgumentError("precision must be 'tc' or 'fp32'")
        _lib.check(self._lib.kws_model_set_precision(self._handle, modes[precision]))
        self.precision = precision

    # -- lifetime
    def close(self):
        if getattr(self, "_handle", None):
            self._lib.kws_model_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._handle

    def num_frames(self, signal_length: int) -> int:
        return int(self._lib.kws_num_frames(self._handle, int(signal_length)))

    def zero_state(self, n_streams: int = 1, numpy: bool = True):
        shape = (self.config.num_layers, n_streams, self.config.hidden_size)
        return np.zeros(shape, np.float32) if numpy else torch.zeros(shape, dtype=torch.float32, device=self.device)

    # -- the deployment call
    def _prep_state(self, state, S):
        L, H = self.config.num_layers, self.config.hidden_size
        st = _tensors.to_device(state, torch.float32, self.device)
        if tuple(st.shape) != (L, S, H):
            raise _lib.InvalidArgumentError("rnn_initial_states must be [%d, %d, %d], got %r" % (L, S, H, tuple(st.shape)))
        return st

    def frame_counts(self, lengths):
        """n_b = max(0, 1 + floor((lengths - fft_size) / hop_size)) frames of rows of ``lengths`` samples, in the
        container type of ``lengths`` (int, list, tuple, numpy or torch): the ``lens`` to give
        ``prediction.decode_batch`` / ``kws_ctc_decode`` for the posteriors of ``forward(pcm, state, lengths=lengths)``."""
        fft, hop = self.config.fft_size, self.config.hop_size
        if isinstance(lengths, torch.Tensor):
            return torch.clamp((lengths - fft) // hop + 1, min=0)
        if isinstance(lengths, np.ndarray):
            return np.maximum((lengths - fft) // hop + 1, 0)
        rule = lambda n: max(0, (int(n) - fft) // hop + 1)
        if isinstance(lengths, (list, tuple)):
            return type(lengths)(rule(n) for n in lengths)
        return rule(lengths)

    def _check_lengths(self, lengths, S: int, L: int):
        """lengths -> int32 CUDA [S].  Host values are validated (0 <= lengths <= L); CUDA values are left to the
        kernels, which clamp them to [0, L] (reading them here would synchronise the stream)."""
        if not _tensors.is_host(lengths):
            if tuple(lengths.shape) != (S,) or lengths.dtype.is_floating_point or lengths.dtype == torch.bool:
                raise _lib.InvalidArgumentError("lengths must be integers [%d], got %s %r"
                                                % (S, lengths.dtype, tuple(lengths.shape)))
            return _tensors.to_device(lengths, torch.int32, self.device)
        a = np.asarray(lengths.numpy() if isinstance(lengths, torch.Tensor) else lengths)
        if a.shape != (S,) or a.dtype.kind not in "iu":
            raise _lib.InvalidArgumentError("lengths must be integers [%d], got %s %r" % (S, a.dtype, a.shape))
        if S and (a.min() < 0 or a.max() > L):
            raise _lib.InvalidArgumentError("lengths must lie in [0, L = %d], got [%d, %d]" % (L, a.min(), a.max()))
        return _tensors.to_device(a.astype(np.int32), torch.int32, self.device)

    def forward(self, inputX, rnn_initial_states, want_logits: bool = False, lengths=None):
        """(pcm, rnn_state) -> (softmax [S,n,C], rnn_state [L,S,H] [, logits]).

        ``lengths [S]`` (host or CUDA integers): valid samples per row.  Row b is then computed as a call on
        ``inputX[b, :lengths[b]]`` alone, bit for bit, on its ``frame_counts(lengths)[b]`` frames: no sample past
        lengths[b] is read, its rows from there on are zero, and its state is the one after its own last frame (the
        incoming state for a row shorter than one frame).  Host lengths must lie in [0, L]."""
        host = _tensors.is_host(inputX)
        pcm = inputX
        is_i16 = (isinstance(pcm, torch.Tensor) and pcm.dtype == torch.int16) or \
                 (not isinstance(pcm, torch.Tensor) and np.asarray(pcm).dtype == np.int16)
        dt = torch.int16 if is_i16 else torch.float32
        x = _tensors.to_device(pcm, dt, self.device)
        if x.dim() == 1:
            x = x.unsqueeze(0)                      # tf.expand_dims(inputX, 0), rnn_ctc.py:134
        if x.dim() != 2:
            raise _lib.InvalidArgumentError("inputX must be [L] or [S, L]")
        S, Lsig = x.shape
        st_in = self._prep_state(rnn_initial_states, S)
        ln = None if lengths is None else self._check_lengths(lengths, S, Lsig)
        n = self.num_frames(Lsig)
        C = self.config.num_classes
        probs = torch.empty((S, max(n, 0), C), dtype=torch.float32, device=self.device)
        logits = torch.empty_like(probs) if want_logits else None
        st_out = torch.empty_like(st_in)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.kws_deploy_forward_lens(
                self._handle, _tensors.ptr(x), _lib.PCM_I16 if is_i16 else _lib.PCM_F32, S, Lsig, x.stride(0) if S > 1 else Lsig,
                _tensors.ptr(ln), _tensors.ptr(st_in), _tensors.ptr(probs), _tensors.ptr(st_out), _tensors.ptr(logits),
                _tensors.stream_ptr(self.device)))
        outs = [probs, st_out] + ([logits] if want_logits else [])
        if host:
            torch.cuda.current_stream(self.device).synchronize()
            outs = [_tensors.to_host(o) for o in outs]
        return tuple(outs)

    __call__ = forward

    def frontend(self, inputX, lengths=None):
        """PCM -> mel frames ``[S, n, M]`` (K1 alone).

        ``lengths [S]`` (host or CUDA integers, host values in [0, L]): valid samples per row; rows
        ``< frame_counts(lengths)[b]`` are bit for bit those of ``frontend(inputX[b, :lengths[b]])``, the rest zero."""
        host = _tensors.is_host(inputX)
        is_i16 = (isinstance(inputX, torch.Tensor) and inputX.dtype == torch.int16) or \
                 (not isinstance(inputX, torch.Tensor) and np.asarray(inputX).dtype == np.int16)
        x = _tensors.to_device(inputX, torch.int16 if is_i16 else torch.float32, self.device)
        if x.dim() == 1:
            x = x.unsqueeze(0)
        if x.dim() != 2:
            raise _lib.InvalidArgumentError("inputX must be [L] or [S, L]")
        S, Lsig = x.shape
        ln = None if lengths is None else self._check_lengths(lengths, S, Lsig)
        n = max(self.num_frames(Lsig), 0)
        mel = torch.empty((S, n, self.config.n_mel), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.kws_frontend_mel_lens(self._handle, _tensors.ptr(x), _lib.PCM_I16 if is_i16 else _lib.PCM_F32,
                                                       S, Lsig, x.stride(0) if S > 1 else Lsig, _tensors.ptr(ln),
                                                       _tensors.ptr(mel), _tensors.stream_ptr(self.device)))
        if host:
            torch.cuda.current_stream(self.device).synchronize()
            return _tensors.to_host(mel)
        return mel

    def run_mel(self, mel, rnn_initial_states, seq_len=None, want_logits: bool = False):
        """(mel frames, rnn_state) -> (softmax, rnn_state [, logits])  (rnn_ctc.py:150-153)."""
        host = _tensors.is_host(mel)
        x = _tensors.to_device(mel, torch.float32, self.device)
        if x.dim() == 2:
            x = x.unsqueeze(0)
        if x.dim() != 3 or x.shape[2] != self.config.n_mel:
            raise _lib.InvalidArgumentError("mel must be [n, %d] or [S, n, %d]" % (self.config.n_mel, self.config.n_mel))
        S, n, _ = x.shape
        st_in = self._prep_state(rnn_initial_states, S)
        sl = None if seq_len is None else _tensors.to_device(seq_len, torch.int32, self.device)
        if sl is not None and tuple(sl.shape) != (S,):
            raise _lib.InvalidArgumentError("seq_len must be [%d], got %r" % (S, tuple(sl.shape)))
        C = self.config.num_classes
        probs = torch.empty((S, n, C), dtype=torch.float32, device=self.device)
        logits = torch.empty_like(probs) if want_logits else None
        st_out = torch.empty_like(st_in)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.kws_gru_forward(self._handle, _tensors.ptr(x), S, n, _tensors.ptr(sl),
                                                 _tensors.ptr(st_in), _tensors.ptr(probs), _tensors.ptr(st_out),
                                                 _tensors.ptr(logits), _tensors.stream_ptr(self.device)))
        outs = [probs, st_out] + ([logits] if want_logits else [])
        if host:
            torch.cuda.current_stream(self.device).synchronize()
            outs = [_tensors.to_host(o) for o in outs]
        return tuple(outs)

    # -- sess.run shim with the frozen graph's tensor names (main.py:339-342, detector.py:190-193)
    def run(self, fetches: Sequence[str], feed_dict: dict):
        single = isinstance(fetches, str)
        names = [fetches] if single else list(fetches)
        known = {SOFTMAX, RNN_STATES, LOGIT}
        for nme in names:
            if nme not in known:
                raise _lib.InvalidArgumentError("unknown fetch %r; the frozen graph exposes %s" % (nme, sorted(known)))
        if INPUT_X not in feed_dict or INITIAL_STATES not in feed_dict:
            raise _lib.InvalidArgumentError("feed_dict must hold %r and %r" % (INPUT_X, INITIAL_STATES))
        outs = self.forward(feed_dict[INPUT_X], feed_dict[INITIAL_STATES], want_logits=LOGIT in names)
        by_name = {SOFTMAX: outs[0], RNN_STATES: outs[1]}
        if LOGIT in names:
            by_name[LOGIT] = outs[2]
        res = [by_name[nme] for nme in names]
        return res[0] if single else res
