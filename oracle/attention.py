"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the attention_ctc deployment forward pass.

Follows models/attention_ctc.py:28-128 (self_attention, feed_forward, inference) and :215-274 (DeployModel) with
the shipped config (config/attention_config.py: n_mel 60, combine_frame 2, hidden 128, 8 heads, 3 layers, FFN 512,
use_relu True).  TensorFlow 1.x semantics restated from its published behaviour:
  * tf.layers.conv2d with a (1,1) kernel = per-position dense layer with bias (kernel [1,1,in,out]);
  * tf.contrib.layers.layer_norm of that era: mean/variance over ALL non-batch axes of the [B,T,N] tensor
    (begin_norm_axis=1), gamma/beta per channel (begin_params_axis=-1), variance_epsilon 1e-12;
  * no padding mask anywhere; softmax over all T' keys.
PARITY UNPINNED: TensorFlow cannot be installed here and the reference has no fixture for this model.
Only tests/, smoke() and bench.py may import this module.
"""
from dataclasses import dataclass, field
from typing import List

import numpy as np

from . import posenc

HIDDEN, HEADS, LAYERS, FFN, COMBINE, CLASSES = 128, 8, 3, 512, 2, 6


@dataclass
class AttentionWeights:
    mel_basis: np.ndarray = None          # [201, M]
    w_in: np.ndarray = None               # input_linear_trans kernel [combine*M, N]
    b_in: np.ndarray = None
    w_qkv: List[np.ndarray] = field(default_factory=list)   # [N, 3N]
    b_qkv: List[np.ndarray] = field(default_factory=list)
    ln1_g: List[np.ndarray] = field(default_factory=list)   # layer_norm after attention (gamma, beta [N])
    ln1_b: List[np.ndarray] = field(default_factory=list)
    w_ff1: List[np.ndarray] = field(default_factory=list)   # conv1 [N, F]
    b_ff1: List[np.ndarray] = field(default_factory=list)
    w_ff2: List[np.ndarray] = field(default_factory=list)   # conv2 [F, N]
    b_ff2: List[np.ndarray] = field(default_factory=list)
    ln2_g: List[np.ndarray] = field(default_factory=list)
    ln2_b: List[np.ndarray] = field(default_factory=list)
    w_out: np.ndarray = None              # output_linear_trans [N, C]
    b_out: np.ndarray = None


def init_weights(seed=4321, n_mel=60, mel_basis=None, combine=COMBINE, layers=LAYERS, ffn=FFN,
                 classes=CLASSES) -> AttentionWeights:
    """Random weights: glorot-uniform kernels (tf.layers.conv2d default) with small random biases and
    non-trivial layer-norm parameters so that every term of the graph is exercised.  The defaults are the
    shipped config; other values give the weights of any config kws_attention_create accepts."""
    from .model import slaney_mel_basis
    rng = np.random.default_rng(seed)

    def glorot(i, o):
        lim = np.sqrt(6.0 / (i + o))
        return rng.uniform(-lim, lim, (i, o)).astype(np.float32)

    w = AttentionWeights()
    w.mel_basis = (slaney_mel_basis(n_mels=n_mel).T if mel_basis is None else mel_basis).astype(np.float32)
    w.w_in = glorot(combine * n_mel, HIDDEN)
    w.b_in = (rng.standard_normal(HIDDEN) * 0.05).astype(np.float32)
    for _ in range(layers):
        w.w_qkv.append(glorot(HIDDEN, 3 * HIDDEN))
        w.b_qkv.append((rng.standard_normal(3 * HIDDEN) * 0.05).astype(np.float32))
        w.ln1_g.append((1 + 0.1 * rng.standard_normal(HIDDEN)).astype(np.float32))
        w.ln1_b.append((0.1 * rng.standard_normal(HIDDEN)).astype(np.float32))
        w.w_ff1.append(glorot(HIDDEN, ffn))
        w.b_ff1.append((rng.standard_normal(ffn) * 0.05).astype(np.float32))
        w.w_ff2.append(glorot(ffn, HIDDEN))
        w.b_ff2.append((rng.standard_normal(HIDDEN) * 0.05).astype(np.float32))
        w.ln2_g.append((1 + 0.1 * rng.standard_normal(HIDDEN)).astype(np.float32))
        w.ln2_b.append((0.1 * rng.standard_normal(HIDDEN)).astype(np.float32))
    w.w_out = glorot(HIDDEN, classes)
    w.b_out = (rng.standard_normal(classes) * 0.05).astype(np.float32)
    return w


def combine_frames(mel, combine=COMBINE):
    """models/attention_ctc.py:77-90: pad with (combine - T % combine) zero frames -- a full extra group when
    T is already a multiple -- and fold `combine` frames into one row.  T' = T // combine + 1."""
    B, T, M = mel.shape
    pad = combine - T % combine
    x = np.concatenate([mel, np.zeros((B, pad, M), mel.dtype)], axis=1)
    return x.reshape(B, -1, M * combine)


def layer_norm(x, gamma, beta, eps=1e-12):
    """tf.contrib.layers.layer_norm (TF 1.x): moments over all non-batch axes, per-channel scale/offset."""
    mean = x.mean(axis=(1, 2), keepdims=True)
    var = ((x - mean) ** 2).mean(axis=(1, 2), keepdims=True)
    return (x - mean) / np.sqrt(var + eps) * gamma + beta


def self_attention(x, w_qkv, b_qkv, heads=HEADS):
    """models/attention_ctc.py:28-58."""
    B, T, N = x.shape
    qkv = x @ w_qkv + b_qkv
    q, k, v = np.split(qkv, 3, axis=2)
    d = N // heads
    q = q.reshape(B, T, heads, d).transpose(0, 2, 1, 3)
    k = k.reshape(B, T, heads, d).transpose(0, 2, 1, 3)
    v = v.reshape(B, T, heads, d).transpose(0, 2, 1, 3)
    a = q @ k.transpose(0, 1, 3, 2) / np.sqrt(d)
    a = a - a.max(axis=-1, keepdims=True)
    a = np.exp(a)
    a = a / a.sum(axis=-1, keepdims=True)
    o = a @ v                                          # [B, h, T, d]
    return o.transpose(0, 2, 1, 3).reshape(B, T, N)


def mel_forward(mel, w: AttentionWeights, dtype=np.float32, use_relu=True, combine=COMBINE):
    """inference() + softmax: mel [B, T, M] -> (softmax [B, T', C], logits).  Layers, FFN width and classes
    follow the weights."""
    f = lambda a: np.asarray(a).astype(dtype)
    x = combine_frames(f(mel), combine)
    x = x @ f(w.w_in) + f(w.b_in)                      # input_linear_trans (:92-95)
    Tp = x.shape[1]
    x = x + f(posenc.positional_encoding(Tp, HIDDEN))  # :96-98
    for l in range(len(w.w_qkv)):
        a = self_attention(x, f(w.w_qkv[l]), f(w.b_qkv[l]))
        y = layer_norm(a + x, f(w.ln1_g[l]), f(w.ln1_b[l]))                       # :111-112
        ff = np.maximum(y @ f(w.w_ff1[l]) + f(w.b_ff1[l]), 0) @ f(w.w_ff2[l]) + f(w.b_ff2[l])   # :61-70
        x = layer_norm(ff + y, f(w.ln2_g[l]), f(w.ln2_b[l]))                      # :118-120
    logits = x @ f(w.w_out) + f(w.b_out)               # output_linear_trans (:122-125)
    if use_relu:
        logits = np.maximum(logits, 0)                 # :126-127
    z = logits - logits.max(axis=-1, keepdims=True)
    e = np.exp(z)
    return (e / e.sum(axis=-1, keepdims=True)).astype(dtype), logits.astype(dtype)


def deploy_forward(pcm, w: AttentionWeights, dtype=np.float32):
    """DeployModel (:215-274) batched over equal-length utterances: pcm [B, L] float (scaled by 2^-15)."""
    from . import model as om
    pcm = np.asarray(pcm)
    if pcm.ndim == 1:
        pcm = pcm[None]
    mel = om.melspec(om.linearspec(om.frame(pcm.astype(dtype)), dtype), w.mel_basis, dtype)
    return mel_forward(mel, w, dtype)
