"""Oracle (TEST INFRASTRUCTURE ONLY): numpy restatement of the rnn_ctc deployment graph.

PARITY UNPINNED for this file: TensorFlow 1.x / librosa are absent (see
oracle/__init__.py).  Every function cites the reference lines it follows.

All functions take ``dtype`` -- ``np.float32`` reproduces the reference's fp32
graph (every intermediate rounded to fp32 like TF's CPU kernels),
``np.float64`` is the high-precision master used to bound rounding noise.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional, Tuple

import numpy as np

# constants of the shipped deployment config (config/rnn_config.py:57-65,76-84)
SAMPLE_RATE = 16000
FFT_SIZE = 400
HOP_SIZE = 160
FMIN = 300.0
FMAX = 8000.0
HIDDEN = 128
NUM_LAYERS = 2
NUM_CLASSES = 6
N_BINS = FFT_SIZE // 2 + 1


# --------------------------------------------------------------------------
# mel filterbank: librosa.filters.mel(sr, n_fft, n_mels, fmin, fmax) with its
# defaults of that era (htk=False -> Slaney scale, norm=1 -> area normalised).
# Call sites: models/rnn_ctc.py:139-144, detector.py:126-129, reader.py:33-38.
# librosa is a third-party dependency that is not vendored and not pinned by
# the reference (no requirements file); this restates its published algorithm.
# --------------------------------------------------------------------------
def _hz_to_mel_slaney(f):
    f = np.asarray(f, dtype=np.float64)
    f_sp = 200.0 / 3.0
    mels = f / f_sp
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = np.log(6.4) / 27.0
    with np.errstate(divide="ignore", invalid="ignore"):
        log_part = min_log_mel + np.log(np.maximum(f, 1e-300) / min_log_hz) / logstep
    return np.where(f >= min_log_hz, log_part, mels)


def _mel_to_hz_slaney(m):
    m = np.asarray(m, dtype=np.float64)
    f_sp = 200.0 / 3.0
    freqs = f_sp * m
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = np.log(6.4) / 27.0
    return np.where(m >= min_log_mel, min_log_hz * np.exp(logstep * (m - min_log_mel)), freqs)


def slaney_mel_basis(sr=SAMPLE_RATE, n_fft=FFT_SIZE, n_mels=40, fmin=FMIN, fmax=FMAX):
    """``librosa.filters.mel`` -> ``[n_mels, 1 + n_fft//2]`` float64."""
    n_bins = 1 + n_fft // 2
    fftfreqs = np.linspace(0.0, float(sr) / 2.0, n_bins)
    mel_pts = np.linspace(_hz_to_mel_slaney(fmin), _hz_to_mel_slaney(fmax), n_mels + 2)
    mel_f = _mel_to_hz_slaney(mel_pts)
    fdiff = np.diff(mel_f)
    ramps = mel_f[:, None] - fftfreqs[None, :]
    weights = np.zeros((n_mels, n_bins), dtype=np.float64)
    for i in range(n_mels):
        lower = -ramps[i] / fdiff[i]
        upper = ramps[i + 2] / fdiff[i + 1]
        weights[i] = np.maximum(0.0, np.minimum(lower, upper))
    enorm = 2.0 / (mel_f[2:n_mels + 2] - mel_f[:n_mels])
    weights *= enorm[:, None]
    return weights


# --------------------------------------------------------------------------
# weights container (layout == the TF variables' own layout, SURVEY.md 8f-3)
# --------------------------------------------------------------------------
@dataclass
class Weights:
    """rnn_ctc deployment parameters in the TF checkpoint layout.

    ``gates_kernel[l]``: ``[in_l + H, 2H]`` rows = concat(x, h), cols = r | u
    ``cand_kernel[l]`` : ``[in_l + H, H]``  rows = concat(x, r*h)
    ``fc_w``           : ``[H, C]`` (weightsClasses), ``fc_b``: ``[C]``
    ``mel_basis``      : ``[201, M]`` (= librosa mel(...).T, rnn_ctc.py:139-146)
    """
    mel_basis: np.ndarray
    gates_kernel: List[np.ndarray] = field(default_factory=list)
    gates_bias: List[np.ndarray] = field(default_factory=list)
    cand_kernel: List[np.ndarray] = field(default_factory=list)
    cand_bias: List[np.ndarray] = field(default_factory=list)
    fc_w: np.ndarray = None
    fc_b: np.ndarray = None

    @property
    def n_mel(self):
        return self.mel_basis.shape[1]

    @property
    def hidden(self):
        return self.fc_w.shape[0]

    @property
    def num_layers(self):
        return len(self.gates_kernel)

    @property
    def num_classes(self):
        return self.fc_w.shape[1]


def init_weights(seed=1234, n_mel=40, hidden=HIDDEN, num_layers=NUM_LAYERS,
                 num_classes=NUM_CLASSES, fc_std=1.0) -> Weights:
    """Random-init weights of the reference architecture (SURVEY.md 8d).

    GRU kernels Xavier-normal (models/rnn_ctc.py:230-232), gate bias 1.0 and
    candidate bias 0.0 (TF GRUCell defaults), FC truncated-normal(std 1) clipped
    at 2 sigma and zero bias (models/rnn_ctc.py:265-273).
    """
    rng = np.random.default_rng(seed)
    w = Weights(mel_basis=slaney_mel_basis(n_mels=n_mel).T.astype(np.float32))
    for layer in range(num_layers):
        fan_in = (n_mel if layer == 0 else hidden) + hidden
        std_g = np.sqrt(2.0 / (fan_in + 2 * hidden))
        std_c = np.sqrt(2.0 / (fan_in + hidden))
        w.gates_kernel.append((rng.standard_normal((fan_in, 2 * hidden)) * std_g).astype(np.float32))
        w.gates_bias.append(np.ones(2 * hidden, dtype=np.float32))
        w.cand_kernel.append((rng.standard_normal((fan_in, hidden)) * std_c).astype(np.float32))
        w.cand_bias.append(np.zeros(hidden, dtype=np.float32))
    fc = rng.standard_normal((hidden, num_classes))
    bad = np.abs(fc) > 2.0
    while bad.any():                     # truncated_normal resamples beyond 2 sigma
        fc[bad] = rng.standard_normal(int(bad.sum()))
        bad = np.abs(fc) > 2.0
    w.fc_w = (fc * fc_std).astype(np.float32)
    w.fc_b = np.zeros(num_classes, dtype=np.float32)
    return w


# --------------------------------------------------------------------------
# front end
# --------------------------------------------------------------------------
def num_frames(signal_length: int, frame_length=FFT_SIZE, frame_step=HOP_SIZE) -> int:
    """utils/stft.py:60-61 -- ``1 + floor((L - frame_length) / frame_step)``."""
    return 1 + int(np.floor((signal_length - frame_length) / frame_step))


def frame(signal: np.ndarray, frame_length=FFT_SIZE, frame_step=HOP_SIZE) -> np.ndarray:
    """utils/stft.py:27-81 ``tf_frame``: ``[S, L] -> [S, n, frame_length]``.

    Rectangular window, no centring, no padding; the tail that does not fill a
    frame is dropped.
    """
    signal = np.asarray(signal)
    if signal.ndim != 2:
        raise ValueError("expected signal to have rank 2 but was %d" % signal.ndim)
    n = num_frames(signal.shape[1], frame_length, frame_step)
    if n <= 0:
        return np.zeros((signal.shape[0], 0, frame_length), dtype=signal.dtype)
    idx = np.arange(frame_length)[None, :] + frame_step * np.arange(n)[:, None]
    return signal[:, idx]


def linearspec(frames: np.ndarray, dtype=np.float32) -> np.ndarray:
    """models/rnn_ctc.py:137 -- ``abs(rfft(frames, [400]))`` -> ``[S, n, 201]``."""
    spec = np.fft.rfft(frames.astype(dtype), n=FFT_SIZE, axis=-1)
    return np.abs(spec).astype(dtype)


def melspec(lin: np.ndarray, mel_basis: np.ndarray, dtype=np.float32) -> np.ndarray:
    """models/rnn_ctc.py:139-149 -- ``linearspec @ mel_basis[201, M]``."""
    return np.matmul(lin.astype(dtype), mel_basis.astype(dtype)).astype(dtype)


def pcm_to_mel(pcm: np.ndarray, w: Weights, dtype=np.float32) -> np.ndarray:
    """PCM ``[S, L]`` (float, already scaled by 2^-15) -> mel ``[S, n, M]``."""
    return melspec(linearspec(frame(pcm), dtype), w.mel_basis, dtype)


# --------------------------------------------------------------------------
# GRU (TF 1.x GRUCell / MultiRNNCell / dynamic_rnn semantics; SURVEY.md 3.2)
# call sites: models/rnn_ctc.py:179-199 (get_cell), :228-244 (inference1)
# --------------------------------------------------------------------------
def _sigmoid(x):
    return 1.0 / (1.0 + np.exp(-x))


def _operand(a, operand_dtype, dtype):
    """Model of a reduced-precision matmul OPERAND (accumulation stays in ``dtype``): used to emulate the
    tensor-core path's arithmetic (fp16 operands, fp32 accumulate) so the kernel's logic can be checked far
    below the 1e-3 contract tolerance.  ``None`` = the reference's plain fp32 graph."""
    return a if operand_dtype is None else a.astype(operand_dtype).astype(dtype)


def _split_product(x, W, od, dtype):
    """Emulation of the tensor-core path's layer-0 input projection: x = x_hi + x_lo and W = W_hi + W_lo in
    ``od`` (fp16), product = x_hi W_hi + x_lo W_hi + x_hi W_lo accumulated in ``dtype``."""
    xh = _operand(x, od, dtype)
    xl = _operand((x - xh).astype(dtype), od, dtype)
    Wh = _operand(W, od, dtype)
    Wl = _operand((W - Wh).astype(dtype), od, dtype)
    return np.matmul(xh, Wh) + np.matmul(xl, Wh) + np.matmul(xh, Wl)


# The tensor-core kernel's shared-memory plan for layer 0 (gru_tc.cu: gru_tc_smem_bytes, gru_tc_x_buffers,
# gru_tc_can_split; api.cu: the split and fit decisions at model creation).  `cap` is the device's opt-in
# shared-memory limit per block; TC_SMEM_OPTIN_B200 is the B200's (227 KB).
TC_SMEM_OPTIN_B200 = 232448
_TC_TILE_CHUNK = 2048          # one 8-column chunk of a 128-stream fp16 operand tile
_TC_FC_OPERAND = 16 * HIDDEN * 2
_TC_MAX_CLASSES = 8
_TC_NUM_BARS = 11


def tc_smem_bytes(kxw: int, last: bool, nbuf: int) -> int:
    return (768 * (kxw + HIDDEN) + nbuf * (kxw // 8) * _TC_TILE_CHUNK + 4 * 384
            + ((_TC_FC_OPERAND + 4 * (4 * 6 + _TC_MAX_CLASSES) * 128) if last else 0) + _TC_NUM_BARS * 8 + 16)


def tc_x_buffers(kxw: int, last: bool, cap: int = TC_SMEM_OPTIN_B200) -> int:
    """x buffers the kernel keeps for a layer with `kxw` operand columns: 2, 1, or 0 (does not fit)."""
    for nbuf in (2, 1):
        if tc_smem_bytes(kxw, last, nbuf) <= cap:
            return nbuf
    return 0


def tc_layer0_plan(n_mel: int, num_layers: int, cap: int = TC_SMEM_OPTIN_B200) -> Tuple[bool, int]:
    """(split, x buffers) of layer 0 on the tensor-core kernel; 0 buffers: the model runs the fp32 kernel."""
    last = num_layers == 1
    kx = (n_mel + 15) // 16 * 16
    split = n_mel <= 64 and tc_x_buffers(2 * kx, last, cap) > 0
    return split, tc_x_buffers(2 * kx if split else kx, last, cap)


def gru_cell(x, h, gates_kernel, gates_bias, cand_kernel, cand_bias, dtype=np.float32, operand_dtype=None,
             split_x=False):
    """One TF GRUCell step.  NOTE reset gate is applied to h BEFORE the
    candidate matmul (not the cuDNN / torch.nn.GRU formulation).

    ``operand_dtype`` / ``split_x`` only model the tensor-core kernel's operand rounding (test infrastructure
    for a tight logic check); the reference graph is ``operand_dtype=None``."""
    one = dtype(1.0)
    od = operand_dtype
    H = h.shape[1]
    if od is None:
        xh = np.concatenate([x, h], axis=1)
        gate_in = (np.matmul(xh, gates_kernel.astype(dtype)) + gates_bias.astype(dtype)).astype(dtype)
    else:
        in_dim = x.shape[1]
        Wx, Wh = gates_kernel[:in_dim].astype(dtype), gates_kernel[in_dim:].astype(dtype)
        xp = _split_product(x, Wx, od, dtype) if split_x else np.matmul(_operand(x, od, dtype), _operand(Wx, od, dtype))
        gate_in = (xp + np.matmul(_operand(h, od, dtype), _operand(Wh, od, dtype)) + gates_bias.astype(dtype)).astype(dtype)
    gates = _sigmoid(gate_in).astype(dtype)
    r, u = gates[:, :H], gates[:, H:]
    rh = (r * h).astype(dtype)
    if od is None:
        xrh = np.concatenate([x, rh], axis=1)
        cand = (np.matmul(xrh, cand_kernel.astype(dtype)) + cand_bias.astype(dtype)).astype(dtype)
    else:
        in_dim = x.shape[1]
        Wx, Wh = cand_kernel[:in_dim].astype(dtype), cand_kernel[in_dim:].astype(dtype)
        xp = _split_product(x, Wx, od, dtype) if split_x else np.matmul(_operand(x, od, dtype), _operand(Wx, od, dtype))
        cand = (xp + np.matmul(_operand(rh, od, dtype), _operand(Wh, od, dtype)) + cand_bias.astype(dtype)).astype(dtype)
    c = np.tanh(cand).astype(dtype)
    return (u * h + (one - u) * c).astype(dtype)


def gru_forward(x: np.ndarray, state: np.ndarray, w: Weights,
                seq_len: Optional[np.ndarray] = None, dtype=np.float32, operand_dtype=None
                ) -> Tuple[np.ndarray, np.ndarray]:
    """``inference1`` (models/rnn_ctc.py:202-244).

    x ``[S, n, M]``, state ``[layers, S, H]`` -> outputs ``[S, n, H]`` of the
    last layer, final state ``[layers, S, H]``.  ``seq_len`` follows
    ``dynamic_rnn(sequence_length=...)``: for ``t >= seq_len[s]`` the output is
    zero and the state is copied through.
    """
    x = x.astype(dtype)
    S, n, _ = x.shape
    h = [state[l].astype(dtype).copy() for l in range(w.num_layers)]
    out = np.zeros((S, n, w.hidden), dtype=dtype)
    split0 = operand_dtype is not None and tc_layer0_plan(x.shape[2], w.num_layers)[0]
    for t in range(n):
        inp = x[:, t, :]
        live = None if seq_len is None else (t < np.asarray(seq_len))[:, None]
        for l in range(w.num_layers):
            new_h = gru_cell(inp, h[l], w.gates_kernel[l], w.gates_bias[l],
                             w.cand_kernel[l], w.cand_bias[l], dtype, operand_dtype,
                             split_x=(split0 and l == 0))
            if live is not None:
                new_h = np.where(live, new_h, h[l])
            h[l] = new_h
            inp = new_h
        out[:, t, :] = inp if live is None else np.where(live, inp, dtype(0))
    return out, np.stack(h, axis=0)


def fc_logits(rnn_out: np.ndarray, w: Weights, dtype=np.float32) -> np.ndarray:
    """``inference2`` (models/rnn_ctc.py:247-284); relu/clip branch is dead
    because ``use_relu`` ends up False (config/rnn_config.py:83)."""
    S, n, H = rnn_out.shape
    flat = rnn_out.reshape(-1, H).astype(dtype)
    logits = (np.matmul(flat, w.fc_w.astype(dtype)) + w.fc_b.astype(dtype)).astype(dtype)
    return logits.reshape(S, n, w.fc_w.shape[1])


def softmax(logits: np.ndarray, dtype=np.float32) -> np.ndarray:
    """``tf.nn.softmax`` over the last axis (models/rnn_ctc.py:165)."""
    z = logits.astype(dtype)
    z = z - z.max(axis=-1, keepdims=True)
    e = np.exp(z).astype(dtype)
    return (e / e.sum(axis=-1, keepdims=True)).astype(dtype)


def mel_forward(mel: np.ndarray, state: np.ndarray, w: Weights, seq_len=None, dtype=np.float32, operand_dtype=None):
    """(mel frames, rnn_state) -> (softmax, rnn_state, logits); the commented
    mel-input form of the deployment graph (models/rnn_ctc.py:150-153)."""
    out, new_state = gru_forward(mel, state, w, seq_len, dtype, operand_dtype)
    logits = fc_logits(out, w, dtype)
    return softmax(logits, dtype), new_state, logits


def deploy_forward(pcm: np.ndarray, state: np.ndarray, w: Weights, dtype=np.float32, operand_dtype=None):
    """``DeployModel`` (models/rnn_ctc.py:113-166) batched over streams.

    pcm ``[S, L]`` float (or ``[L]``, the reference's batch-1 form), state
    ``[layers, S, H]`` -> softmax ``[S, n, C]``, state, logits ``[S, n, C]``.
    """
    pcm = np.asarray(pcm)
    if pcm.ndim == 1:
        pcm = pcm[None, :]
    mel = pcm_to_mel(pcm.astype(dtype), w, dtype)
    return mel_forward(mel, state, w, None, dtype, operand_dtype)


def pcm16_to_float(x: np.ndarray) -> np.ndarray:
    """detector.py:40-43 ``buf_to_float`` -- int16 LE PCM -> float32 * 2^-15."""
    return (np.float32(1.0 / 32768.0) * np.asarray(x, dtype=np.int16).astype(np.float32)).astype(np.float32)


# --------------------------------------------------------------------------
# the octbit-rewritten deployment graph (graph_octbit.pb: main.py:357-371,
# octbit/octbit_graph.py:218-225, 461-536).  Every MatMul outside cell_0 is an
# OctbitMatMul: gates / candidate of the upper layers and the FC.  The op
# quantises with the min / max of the whole tensor it is called with
# (octbit_mat_mul_op.cc:90-124); the reference deploys at batch 1, so every
# stream below is its own sequence of op calls: [1, in+H] per step for the two
# GRU MatMuls, [n, H] per chunk for the FC (inference2 flattens the frames).
# --------------------------------------------------------------------------
def octize_model(w: Weights, layers=None, fc=True):
    """What GraphRewriter does to the float graph: ``{"gates": {l: (wq, scale, bias)}, "candidate": {...}, "fc": ...}``
    with ``octize_weight_int8_signed`` (octbit_graph.py:191-215); ``scale`` rounded to the fp32 attr."""
    from . import octbit as ooct
    layers = list(range(1, w.num_layers)) if layers is None else list(layers)

    def one(k):
        wq, scale, bias = ooct.octize_weight_int8_signed(k)
        return wq, float(np.float32(scale)), bias.astype(np.float32)

    out = {"gates": {}, "candidate": {}, "fc": None}
    for l in layers:
        out["gates"][l] = one(w.gates_kernel[l])
        out["candidate"][l] = one(w.cand_kernel[l])
    if fc:
        out["fc"] = one(w.fc_w)
    return out


def _octbit_op(x, mat, use_ref=True):
    """One OctbitMatMul call: the unmodified reference kernel (oracle/_ref) when built, else the numpy restatement."""
    from . import cref, octbit as ooct
    wq, scale, bias = mat
    x = np.ascontiguousarray(x, np.float32)
    if use_ref and cref.have_ref():
        return cref.ref_octbit_matmul(x, wq, bias, scale)
    return ooct.octbit_mat_mul(x, wq, scale=np.float32(scale), bias=bias)


def octbit_mel_forward(mel, state, w: Weights, octw, seq_len=None, use_ref=True, trace=None):
    """(mel frames, rnn_state) -> (softmax, rnn_state, logits) of the octbit graph, stream by stream as the
    reference runs it (batch 1).  ``trace``: optional dict filled with the inputs / raw outputs of every op call
    of stream 0 (for op-level checks)."""
    f32 = np.float32
    mel = np.asarray(mel, f32)
    S, n, _ = mel.shape
    L, H, C = w.num_layers, w.hidden, w.num_classes
    new_state = np.array(state, dtype=f32, copy=True)
    probs = np.zeros((S, n, C), f32)
    logits = np.zeros((S, n, C), f32)
    for s in range(S):
        length = n if seq_len is None else int(seq_len[s])
        h = [new_state[l, s].copy() for l in range(L)]
        ys = np.zeros((n, H), f32)
        for t in range(n):
            inp = mel[s, t]
            live = t < length
            for l in range(L):
                if l in octw["gates"]:
                    xh = np.concatenate([inp, h[l]])[None, :]
                    g = _octbit_op(xh, octw["gates"][l], use_ref)[0]
                    gates = _sigmoid((g + w.gates_bias[l]).astype(f32)).astype(f32)
                    r, u = gates[:H], gates[H:]
                    xrh = np.concatenate([inp, (r * h[l]).astype(f32)])[None, :]
                    cpre = _octbit_op(xrh, octw["candidate"][l], use_ref)[0]
                    c = np.tanh((cpre + w.cand_bias[l]).astype(f32)).astype(f32)
                    nh = (u * h[l] + (f32(1) - u) * c).astype(f32)
                    if trace is not None and s == 0:
                        trace.setdefault("steps", []).append(dict(layer=l, t=t, xh=xh[0].copy(), g=g.copy(), xrh=xrh[0].copy(), c=cpre.copy()))
                else:
                    nh = gru_cell(inp[None, :], h[l][None, :], w.gates_kernel[l], w.gates_bias[l], w.cand_kernel[l],
                                  w.cand_bias[l], f32)[0]
                if live:
                    h[l] = nh
                inp = nh
            ys[t] = inp if live else 0
        if octw["fc"] is not None:
            if length > 0:
                lg = _octbit_op(ys[:length], octw["fc"], use_ref)
                logits[s, :length] = (lg + w.fc_b).astype(f32)
            logits[s, length:] = w.fc_b                      # zero rows: q = offset -> (sum - bias) = 0 -> logits = b
        else:
            logits[s] = (ys @ w.fc_w.astype(f32) + w.fc_b).astype(f32)
        probs[s] = softmax(logits[s][None])[0]
        for l in range(L):
            new_state[l, s] = h[l]
    return probs, new_state, logits


def octbit_deploy_forward(pcm, state, w: Weights, octw, use_ref=True):
    pcm = np.asarray(pcm)
    if pcm.ndim == 1:
        pcm = pcm[None, :]
    mel = pcm_to_mel(pcm.astype(np.float32), w, np.float32)
    return octbit_mel_forward(mel, state, w, octw, None, use_ref)
