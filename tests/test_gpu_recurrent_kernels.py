"""GPU: the recurrent kernels step by step against float64 (tests/_gru_ref.py), in every shared-memory regime of the
tensor-core kernel and at the layer, mel and class counts the C-ABI accepts.

- Teacher-forced steps: kws_gru_forward with n = 1 from given states.  Layer 0 is fed the given mel, layer l > 0
  the GPU's own state_out[l - 1], the FC the GPU's last-layer state; every element is held to its own bound.
- Sequences equal their steps: an n-frame call equals n one-frame calls that carry the state, bit for bit.  The
  per-step arithmetic is the same in both forms (the state stays fp32 between steps in both), so any difference
  is a bug: a frame stored in the wrong place, a state reset at a time-chunk boundary, a length applied wrongly.
- Persistent loops: a CTA that runs a second tile must give what a first tile gives (batch independence).
"""
from dataclasses import dataclass

import numpy as np
import pytest

from tests._gru_ref import (EXPF_REL, U, f32_fc, f32_layer_step, octbit_fc_logits, octbit_layer_step, softmax_bound,
                            tc_fc, tc_layer_step, tc_plan, tc_regime)

pytestmark = pytest.mark.gpu

MELS = [1, 3, 16, 17, 32, 33, 41, 48, 49, 64, 65, 80, 81, 96, 97, 127, 128]
TC_CONFIGS = ([(1, m, 6) for m in MELS] + [(2, m, 6) for m in MELS] +
              [(3, 40, 6), (3, 97, 6), (4, 16, 6), (4, 128, 6), (1, 40, 2), (2, 40, 2), (2, 40, 7), (2, 40, 8),
               (2, 40, 9), (2, 40, 16), (1, 24, 16)])
FP32_CONFIGS = [(1, 40, 6), (2, 40, 6), (3, 40, 6), (4, 40, 6), (1, 3, 6), (2, 17, 6), (2, 41, 6), (2, 97, 6),
                (1, 128, 6), (3, 1, 6), (2, 40, 9), (2, 40, 16)]
# (layers, n_mel, converted layers, FC converted)
OCT_CONFIGS = [(1, 40, [], True), (2, 40, [1], True), (3, 40, [1, 2], True), (4, 40, [1, 2, 3], True),
               (3, 40, [1], True), (3, 40, [2], True), (2, 40, [1], False), (3, 41, [1, 2], True)]
SEQ_N = [2, 3, 5, 63, 64, 65, 127, 128, 129, 300]
SEQ_S = [1, 63, 64, 65, 127, 128, 129, 300]
WORST = {}


def _cap():
    import torch
    return int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


def _config(L, M, C):
    from keyword_spotting_b200 import Config

    @dataclass
    class Cfg(Config):
        classes: int = 6

        @property
        def num_classes(self):
            return self.classes

    return Cfg(n_mel=M, num_layers=L, classes=C)


def _weights(L, M, C, seed):
    """Reference init, with gate biases that push some pre-activations past +-20 and over the exponent clamp at 31
    (sigmoid: |z| > 21.5; tanh: |z| > 10.8), and an FC whose logits reach about +-40."""
    from oracle import model as om
    ow = om.init_weights(seed=seed, n_mel=M, num_layers=L, num_classes=C, fc_std=3.5)
    rng = np.random.default_rng(seed + 1)
    for l in range(L):
        ow.gates_bias[l][:6] = np.array([25.0, -25.0, 40.0, -40.0, 21.0, -21.0], np.float32)
        ow.gates_bias[l][128:134] = np.array([25.0, -25.0, 40.0, -40.0, 21.0, -21.0], np.float32)
        ow.cand_bias[l][:4] = np.array([12.0, -12.0, 20.0, -20.0], np.float32)
        ow.gates_bias[l][6:128] += rng.normal(0.0, 1.0, 122).astype(np.float32)
    ow.fc_b = rng.normal(0.0, 2.0, C).astype(np.float32)
    return ow


def _model(ow, L, M, C, precision, octw=None):
    from tests._util import to_product_weights
    from keyword_spotting_b200 import DeployModel
    dm = DeployModel(_config(L, M, C), to_product_weights(ow), device=0, precision=precision)
    if octw is not None:
        dm.set_octbit(octw)
    return dm


def _mel(rng, S, n, M):
    """Mel levels from 0 to about 60 (log-uniform per stream), exact zeros: whole frames and single elements."""
    lev = np.exp(rng.uniform(np.log(1e-3), np.log(60.0), (S, 1, 1)))
    x = (rng.random((S, n, M)) * lev).astype(np.float32)
    x[rng.random((S, n, M)) < 0.1] = 0.0
    x[rng.random((S, n)) < 0.05] = 0.0
    x[0] = 0.0
    return x


def _states(rng, L, S):
    st = rng.uniform(-1.0, 1.0, (L, S, 128)).astype(np.float32)
    st[rng.random((L, S, 128)) < 0.05] = 0.999
    st[rng.random((L, S, 128)) < 0.05] = -0.999
    st[rng.random((L, S, 128)) < 0.05] = 0.0
    st[:, 1 % S] = 0.0
    return st


def _call(dm, x, st_in, seq_len=None, inplace=False):
    """kws_gru_forward -> (probs, state_out, logits) as numpy.  inplace: state_in == state_out."""
    import torch
    from keyword_spotting_b200 import _lib
    S, n, _ = x.shape
    L, C = dm.config.num_layers, dm.config.num_classes
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    sd = torch.from_numpy(np.ascontiguousarray(st_in)).cuda()
    so = sd if inplace else torch.empty_like(sd)
    sl = None if seq_len is None else torch.from_numpy(np.asarray(seq_len, np.int32)).cuda()
    pr = torch.empty((S, n, C), dtype=torch.float32, device="cuda")
    lg = torch.empty_like(pr)
    p = lambda t: 0 if t is None else t.data_ptr()
    _lib.check(dm._lib.kws_gru_forward(dm.handle, p(xd), S, n, p(sl), p(sd), p(pr), p(so), p(lg),
                                       torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return pr.cpu().numpy(), so.cpu().numpy(), lg.cpu().numpy()


def _octw(dm, layers, fc):
    from keyword_spotting_b200 import OctbitModelWeights
    return OctbitModelWeights.from_float(dm.weights, layers=layers, fc=fc)


def _mat(m):
    return (m.weight_q, m.scale, m.bias)


def _note(key, ratio):
    WORST[key] = max(WORST.get(key, 0.0), float(ratio))


def _within(key, got, want, bound):
    err = np.abs(got.astype(np.float64) - want)
    ratio = err / bound
    _note(key, ratio.max())
    bad = np.argwhere(ratio > 1.0)
    assert bad.size == 0, "%s: %d elements out of bound (worst error / bound %.3g), first %r: got %r want %r bound %r" % (
        key, len(bad), ratio.max(), tuple(bad[0]), got[tuple(bad[0])], want[tuple(bad[0])], bound[tuple(bad[0])])


# ================================================================ teacher-forced steps
def _teacher_forced(dm, ow, kind, S, seed, octw=None):
    """One n = 1 call; every layer, the logits and the probabilities against the reference of its back end."""
    L, M, C = ow.num_layers, ow.n_mel, ow.num_classes
    rng = np.random.default_rng(seed)
    x = _mel(rng, S, 1, M)
    st = _states(rng, L, S)
    probs, so, lg = _call(dm, x, st)
    assert np.isfinite(probs).all() and np.isfinite(so).all()
    split0 = tc_plan(M, L, _cap())[0] if kind == "tc" else False
    flagged_total = 0
    for l in range(L):
        inp = x[:, 0] if l == 0 else so[l - 1]
        args = (inp, st[l], ow.gates_kernel[l], ow.gates_bias[l], ow.cand_kernel[l], ow.cand_bias[l])
        if kind == "tc":
            want, bound = tc_layer_step(*args, split=split0 and l == 0)
        elif octw is not None and l in octw.gates:
            want, bound, flagged, quantum = octbit_layer_step(*args, _mat(octw.gates[l]), _mat(octw.candidate[l]))
            flagged_total += int(flagged.sum())
            ok = ~flagged
            _within("octbit h'", so[l][ok], want[ok], bound[ok])
            if flagged.any():
                _within("octbit h' (flagged)", so[l][flagged], want[flagged], bound[flagged] + quantum[flagged])
            continue
        else:
            want, bound = f32_layer_step(*args)
        _within("%s h'" % kind, so[l], want, bound)
    hl = so[L - 1]
    if octw is not None and octw.fc is not None:
        for s in range(S):
            want_lg = octbit_fc_logits(hl[s:s + 1], _mat(octw.fc), ow.fc_b)
            assert np.array_equal(lg[s], want_lg), s               # the op is exact; + b in fp32 as the kernel
        p, dp = softmax_bound(lg[:, 0], np.zeros_like(lg[:, 0]), EXPF_REL, U)
        _within("octbit probs", probs[:, 0], p, dp)
    else:
        want_lg, dlg, p, dp = (tc_fc if kind == "tc" else f32_fc)(hl, ow.fc_w, ow.fc_b)
        name = "octbit" if octw is not None else kind
        _within("%s logits" % name, lg[:, 0], want_lg, dlg)
        _within("%s probs" % name, probs[:, 0], p, dp)
    return flagged_total


@pytest.mark.parametrize("L,M,C", TC_CONFIGS)
def test_tc_teacher_forced_step(L, M, C):
    """The default precision.  Where the tensor-core kernel does not apply (a 1-layer model too wide for shared
    memory, or more than 8 classes) the model runs the fp32 kernel: its output must be that kernel's, bit for bit."""
    ow = _weights(L, M, C, seed=100 + 7 * L + M + C)
    dm = _model(ow, L, M, C, "tc")
    fallback = tc_regime(M, L, _cap()) == "fp32" or C > 8
    if not fallback:
        _teacher_forced(dm, ow, "tc", 256, seed=M * 10 + L)
        return
    ref = _model(ow, L, M, C, "fp32")
    rng = np.random.default_rng(M + L)
    x, st = _mel(rng, 129, 3, M), _states(rng, L, 129)
    for a, b in zip(_call(dm, x, st), _call(ref, x, st)):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    _teacher_forced(dm, ow, "fp32", 256, seed=M * 10 + L)


@pytest.mark.parametrize("L,M,C", FP32_CONFIGS)
def test_fp32_teacher_forced_step(L, M, C):
    ow = _weights(L, M, C, seed=200 + 7 * L + M + C)
    _teacher_forced(_model(ow, L, M, C, "fp32"), ow, "fp32", 256, seed=M * 10 + L + 1)


@pytest.mark.parametrize("L,M,layers,fc", OCT_CONFIGS)
def test_octbit_teacher_forced_step(L, M, layers, fc, capsys):
    """Streams the reference does not flag agree within the float bound; flagged streams (an element of
    [x | r*h] so close to a u8 rounding boundary that the kernel's sigmoid may move it) within one u8 quantum of
    each element that may flip."""
    ow = _weights(L, M, 6, seed=300 + 7 * L + M + len(layers))
    dm = _model(ow, L, M, 6, "fp32")
    octw = _octw(dm, layers, fc)
    dm.set_octbit(octw)
    S = 96
    flagged = _teacher_forced(dm, ow, "fp32", S, seed=M + L + 3, octw=octw)
    frac = flagged / (S * max(1, len(layers)))
    with capsys.disabled():
        print("\n[octbit %d layers, converted %r, fc %s] flagged streams %.1f%%" % (L, layers, fc, 100 * frac))
    assert frac <= 0.25


def test_regimes_reached():
    """Each shared-memory regime of layer 0 (split or not, 2 or 1 x buffers, or the fp32 fallback), below other
    layers and as the only layer, is run by some configuration above."""
    cap = _cap()
    seen = {(L == 1, tc_regime(M, L, cap)) for L, M, C in TC_CONFIGS if C <= 8}
    want = {(only, r) for only in (False, True) for r in ("split2", "split1", "unsplit2", "unsplit1")} | {(True, "fp32")}
    assert want <= seen, sorted(want - seen)


# ================================================================ sequences equal their steps
def _lens(rng, S, n):
    """seq_len: the first warp of each tile live to the end, then 0, 1, n-1, n, > n and values at and around
    64 / 128 next to each other (mixed warps), then random."""
    lens = np.full(S, n + 3, np.int32)
    special = [0, 1, n - 1, n, n + 1, 63, 64, 65, 127, 128, 129, 2, n // 2]
    for s in range(S):
        if s % 128 >= 32:
            i = (s % 128) - 32
            lens[s] = special[i] if i < len(special) else rng.integers(0, n + 2)
    return np.maximum(lens, 0)


def _sequence_vs_steps(dm, S, n, seed, use_len, octw=None):
    L, M = dm.config.num_layers, dm.config.n_mel
    rng = np.random.default_rng(seed)
    x = _mel(rng, S, n, M)
    st = _states(rng, L, S)
    lens = _lens(rng, S, n) if use_len else None
    probs, so, lg = _call(dm, x, st, lens)
    _, so_in, _ = _call(dm, x, st, lens, inplace=True)
    assert np.array_equal(so.view(np.uint32), so_in.view(np.uint32)), "state_in == state_out"
    cur = st
    ys = np.zeros((S, n, 128), np.float32)
    step_probs = np.zeros_like(probs)
    for t in range(n):
        sl = None if lens is None else (t < lens).astype(np.int32)
        prev = cur
        p1, cur, _ = _call(dm, x[:, t:t + 1], cur, sl)
        step_probs[:, t] = p1[:, 0]
        live = np.ones(S, bool) if lens is None else t < lens
        # dynamic_rnn: a frame past the stream's length carries every layer's state through unchanged
        assert np.array_equal(cur[:, ~live].view(np.uint32), prev[:, ~live].view(np.uint32)), "state moved past seq_len"
        ys[live, t] = cur[L - 1][live]
    bad = np.argwhere(so.view(np.uint32) != cur.view(np.uint32))
    assert bad.size == 0, "state differs from the steps' at (layer, stream, unit) %r of %d" % (tuple(bad[0]), len(bad))
    if octw is not None and octw.fc is not None:
        # the octbit FC's range is per call: its logits against the op on this stream's frames, bit for bit
        for s in range(S):
            ln = n if lens is None else min(int(lens[s]), n)
            if ln > 0:
                assert np.array_equal(lg[s, :ln], octbit_fc_logits(ys[s, :ln], _mat(octw.fc), dm.weights.fc_b)), s
            assert np.array_equal(lg[s, ln:], np.broadcast_to(dm.weights.fc_b, lg[s, ln:].shape)), s
        return
    bad = np.argwhere(probs.view(np.uint32) != step_probs.view(np.uint32))
    assert bad.size == 0, "probs differ from the steps' at (stream, frame, class) %r of %d" % (tuple(bad[0]), len(bad))


@pytest.mark.parametrize("precision", ["tc", "fp32"])
@pytest.mark.parametrize("S", SEQ_S)
def test_deployment_model_sequence_equals_steps(precision, S):
    """The deployment shape (2 layers, 40 mels, 6 classes) over every length; n >= 128 with S <= 300 runs the
    tensor-core kernel's two-stream layer pipeline in 64-frame chunks."""
    ow = _weights(2, 40, 6, seed=11)
    dm = _model(ow, 2, 40, 6, precision)
    for i, n in enumerate(SEQ_N):
        _sequence_vs_steps(dm, S, n, seed=1000 * S + n, use_len=(i % 2 == 1) or n >= 128)
    if S >= 64:
        _sequence_vs_steps(dm, S, 129, seed=7 * S, use_len=False)
        _sequence_vs_steps(dm, S, 300, seed=9 * S, use_len=True)


SEQ_CONFIGS = ([("tc", L, M, C) for L, M, C in TC_CONFIGS if not (L == 2 and M == 40 and C == 6)] +
               [("fp32", L, M, C) for L, M, C in FP32_CONFIGS if not (L == 2 and M == 40 and C == 6)])


@pytest.mark.parametrize("precision,L,M,C", SEQ_CONFIGS)
def test_sequence_equals_steps(precision, L, M, C):
    ow = _weights(L, M, C, seed=400 + L + M + C)
    dm = _model(ow, L, M, C, precision)
    _sequence_vs_steps(dm, 129, 129 if L == 2 else 65, seed=L * 1000 + M, use_len=True)
    _sequence_vs_steps(dm, 65, 5, seed=L * 1000 + M + 1, use_len=False)


@pytest.mark.parametrize("L,M,layers,fc", OCT_CONFIGS)
def test_octbit_sequence_equals_steps(L, M, layers, fc):
    """The octbit layers' state bit for bit; the FC (per-call range) against the op on the stream's frames."""
    ow = _weights(L, M, 6, seed=500 + L + M + len(layers))
    dm = _model(ow, L, M, 6, "fp32")
    octw = _octw(dm, layers, fc)
    dm.set_octbit(octw)
    _sequence_vs_steps(dm, 65, 67, seed=L + M, use_len=True, octw=octw)
    _sequence_vs_steps(dm, 33, 5, seed=L + M + 1, use_len=False, octw=octw)


# ================================================================ persistent loops
def _batch_independence(dm, S, n, seed):
    """S streams replay B distinct inputs; every stream must give, bit for bit, what its representative gives.
    Representatives sit in the first tiles, so the second tile of each CTA is checked against a first tile."""
    L, M = dm.config.num_layers, dm.config.n_mel
    B = 97
    rng = np.random.default_rng(seed)
    xb, sb = _mel(rng, B, n, M), _states(rng, L, B)
    idx = rng.integers(0, B, S)
    idx[:B] = np.arange(B)
    x = np.ascontiguousarray(xb[idx])
    st = np.ascontiguousarray(sb[:, idx])
    lens = rng.integers(0, n + 1, B).astype(np.int32)[idx]
    probs, so, _ = _call(dm, x, st, lens)
    assert np.array_equal(probs.view(np.uint32), probs[idx].view(np.uint32))
    assert np.array_equal(so.view(np.uint32), so[:, idx].view(np.uint32))


def test_fp32_second_tile_per_cta():
    """gru.cu: 148 CTAs of 64 streams; S > 9,472 gives some CTA a second tile."""
    ow = _weights(2, 40, 6, seed=21)
    dm = _model(ow, 2, 40, 6, "fp32")
    _batch_independence(dm, 148 * 64 + 1000, 3, seed=5)


def test_octbit_second_pass_per_cta():
    """gru_octbit.cu: 3 x 148 CTAs of 32 streams; S > 14,208 gives some CTA a second part."""
    ow = _weights(2, 40, 6, seed=22)
    dm = _model(ow, 2, 40, 6, "fp32")
    dm.set_octbit(_octw(dm, [1], True))
    _batch_independence(dm, 3 * 148 * 32 + 1500, 3, seed=6)


# ================================================================ calls without frames
@pytest.mark.parametrize("backend", ["tc", "fp32", "octbit"])
def test_zero_frame_call_passes_the_state_through(backend):
    """kws_gru_forward with n = 0 and state_out != state_in: state_out is state_in, bit for bit."""
    L, M = 2, 40
    ow = _weights(L, M, 6, seed=23)
    dm = _model(ow, L, M, 6, "tc" if backend == "tc" else "fp32")
    if backend == "octbit":
        dm.set_octbit(_octw(dm, [1], True))
    rng = np.random.default_rng(24)
    for S in (1, 65, 300):
        st = _states(rng, L, S)
        _, so, _ = _call(dm, np.zeros((S, 0, M), np.float32), st)
        assert np.array_equal(so.view(np.uint32), st.view(np.uint32)), S


def test_report_worst_ratios(capsys):
    """Worst error / bound of every back end and step quantity seen by the tests above (run after them)."""
    with capsys.disabled():
        print("\n[recurrent kernels] worst |error| / bound:")
        for k in sorted(WORST):
            print("  %-24s %.3g" % (k, WORST[k]))
