"""CPU: the float64 recurrent reference of tests/_gru_ref.py -- its values without rounding, the tensor-core kernel's
layer-0 shared-memory plan, and its bounds on constructed worst cases."""
import numpy as np
import pytest

from tests import _gru_ref as gr
from oracle import model as om

f32 = np.float32
LOG2E32 = f32(1.4426950408889634)


def _layer(rng, M, seed=0):
    w = om.init_weights(seed=seed, n_mel=M, num_layers=2)
    x = (rng.random((16, M)) * 30.0).astype(f32)
    h = rng.uniform(-1, 1, (16, 128)).astype(f32)
    return w, x, h


@pytest.mark.parametrize("split", [False, True])
def test_reference_without_rounding_is_gru_cell(monkeypatch, split):
    """With the operand roundings switched off, each back end's step is oracle.model.gru_cell in float64."""
    rng = np.random.default_rng(1)
    w, x, h = _layer(rng, 40)
    want = om.gru_cell(x.astype(np.float64), h.astype(np.float64), w.gates_kernel[0], w.gates_bias[0],
                       w.cand_kernel[0], w.cand_bias[0], dtype=np.float64)
    got, _ = gr.f32_layer_step(x, h, w.gates_kernel[0], w.gates_bias[0], w.cand_kernel[0], w.cand_bias[0])
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-13)
    monkeypatch.setattr(gr, "rn16", lambda a: np.asarray(a, np.float64))
    monkeypatch.setattr(gr, "split16", lambda a: (np.asarray(a, np.float64), np.zeros(np.shape(a))))
    got, _ = gr.tc_layer_step(x, h, w.gates_kernel[0], w.gates_bias[0], w.cand_kernel[0], w.cand_bias[0], split=split)
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-13)


def test_tc_step_models_the_split():
    """Layer 0 split: x_hi W_hi + x_lo W_hi + x_hi W_lo is within 2^-20 relative of fp32 operands; unsplit is not."""
    rng = np.random.default_rng(2)
    w, x, h = _layer(rng, 40)
    exact, _ = gr.f32_layer_step(x, h, w.gates_kernel[0], w.gates_bias[0], w.cand_kernel[0], w.cand_bias[0])
    a, _ = gr.tc_layer_step(x, h, w.gates_kernel[0], w.gates_bias[0], w.cand_kernel[0], w.cand_bias[0], split=True)
    b, _ = gr.tc_layer_step(x, h, w.gates_kernel[0], w.gates_bias[0], w.cand_kernel[0], w.cand_bias[0], split=False)
    assert np.abs(a - exact).max() < 3e-3 and np.abs(a - exact).max() < 0.5 * np.abs(b - exact).max()


def test_layer0_plan_at_the_b200_limit():
    """The table of the regimes at the 227 KB opt-in limit: (split, x buffers) below other layers / as the only one."""
    cap = om.TC_SMEM_OPTIN_B200
    rows = [(1, 32, "split2", "split2"), (33, 48, "split2", "split1"), (49, 64, "split1", "unsplit2"),
            (65, 80, "unsplit2", "unsplit2"), (81, 96, "unsplit2", "unsplit1"), (97, 128, "unsplit1", "fp32")]
    for lo, hi, below, only in rows:
        for M in range(lo, hi + 1):
            assert gr.tc_regime(M, 2, cap) == below, M
            assert gr.tc_regime(M, 3, cap) == below, M
            assert gr.tc_regime(M, 1, cap) == only, M


def test_oracle_emulation_splits_as_the_kernel():
    """oracle.model.gru_forward's tensor-core emulation splits layer 0 exactly where the kernel does: a 1-layer
    model of 49-64 mels is not split."""
    rng = np.random.default_rng(3)
    for L, M, split in [(1, 56, False), (2, 56, True), (1, 40, True), (2, 80, False)]:
        w = om.init_weights(seed=4, n_mel=M, num_layers=L)
        x = (rng.random((4, 1, M)) * 40).astype(f32)
        st = np.zeros((L, 4, 128), f32)
        _, got = om.gru_forward(x, st, w, dtype=np.float64, operand_dtype=np.float16)
        want = om.gru_cell(x[:, 0].astype(np.float64), st[0].astype(np.float64), w.gates_kernel[0], w.gates_bias[0],
                           w.cand_kernel[0], w.cand_bias[0], np.float64, np.float16, split_x=split)
        assert np.array_equal(got[0], want), (L, M)


def test_accum_bound_worst_case():
    """Sequential fp32 sums built to lose the most (a large first term, then terms of half an ulp) stay inside."""
    for n in (8, 64, 272):
        terms = np.full(n, f32(2.0 ** -24) * f32(1.0 - 2.0 ** -20), f32)
        terms[0] = 1.0
        acc = f32(0)
        for t in terms:
            acc = f32(acc + t)
        exact = terms.astype(np.float64).sum()
        assert abs(float(acc) - exact) <= gr.accum_bound(n, np.abs(terms.astype(np.float64)).sum())
        assert abs(float(acc) - exact) >= 0.4 * (n - 1) * 2.0 ** -24      # it is a worst case


def _recip4(e_vals, ex2_err, rcp_err):
    """recip4_1p_exp2 in fp32 with ex2 and rcp off by the given relative errors."""
    e = np.minimum(np.asarray(e_vals, f32), f32(31.0))
    E = (np.exp2(e.astype(np.float64)) * (1 + ex2_err)).astype(f32)
    d = (E + f32(1)).astype(f32)
    pp = np.array([d[0] * d[2], d[1] * d[3]], f32)
    r = f32(np.float64(1.0) / np.float64(f32(pp[0] * pp[1])) * (1 + rcp_err))
    rinv = np.array([r * pp[1], r * pp[0]], f32)
    return np.array([rinv[0] * d[2], rinv[1] * d[3], rinv[0] * d[0], rinv[1] * d[1]], f32)


@pytest.mark.parametrize("mul", [-1.4426950408889634, 2 * 1.4426950408889634])
def test_tc_activation_bound_worst_case(mul):
    """The shared-reciprocal activation with ex2 / rcp at their error limits in either direction, the accumulator off
    by its bound, and exponents past the clamp at 31, stays inside tc_act_bound."""
    rng = np.random.default_rng(5)
    m32 = f32(mul)
    worst = 0.0
    for _ in range(400):
        a = rng.normal(0, 8, 4)
        a[rng.integers(0, 4)] = rng.choice([-40.0, 40.0, 25.0, -25.0])
        b = rng.normal(0, 2, 4)
        dacc = np.abs(a) * 1e-5
        want, bound = gr.tc_act_bound(a, b, dacc, mul)
        for sgn in (-1, 1):
            ak = (a + sgn * dacc).astype(f32)
            nb = (b.astype(f32) * m32).astype(f32)
            e = (ak.astype(np.float64) * np.float64(m32) + nb).astype(f32)          # fma: one rounding
            for ex2e in (-gr.EX2_REL, gr.EX2_REL):
                for rcpe in (-gr.RCP_REL, gr.RCP_REL):
                    got = _recip4(e, ex2e, rcpe).astype(np.float64)
                    ratio = np.abs(got - want) / bound
                    worst = max(worst, ratio.max())
    assert worst <= 1.0, worst
    assert worst > 0.05, worst                                          # and the bound is not vacuous


def test_f32_activation_bounds_worst_case():
    rng = np.random.default_rng(6)
    z = np.concatenate([rng.normal(0, 6, 2000), [0.0, 30.0, -30.0, 1e-6]])
    dacc = np.abs(z) * 1e-6
    for fn, exact in ((gr.f32_sigmoid, None), (gr.f32_tanh, None)):
        want, bound = fn(z, np.zeros_like(z), dacc)
        for sgn in (-1, 1):
            zk = (z + sgn * dacc).astype(f32)
            for err in (-gr.EXPF_REL, gr.EXPF_REL):
                if fn is gr.f32_sigmoid:
                    ex = (np.exp(-zk.astype(np.float64)) * (1 + err)).astype(f32)
                    got = (f32(1) / (f32(1) + ex)).astype(np.float64)
                else:
                    got = (np.tanh(zk.astype(np.float64)) * (1 + err)).astype(f32).astype(np.float64)
                assert (np.abs(got - want) <= bound).all()


def test_softmax_bound_worst_case():
    """Logits moved by their bound in the worst direction (the class up, every other down) and exponentials at the
    error limit stay inside softmax_bound."""
    rng = np.random.default_rng(7)
    lg = rng.normal(0, 15, (200, 6))
    lg[:, 0] = 40.0
    dlg = np.full_like(lg, 1e-5)
    p, dp = gr.softmax_bound(lg, dlg, gr.EX2_REL, gr.RCP_REL + gr.U)
    for c in range(6):
        for sgn in (-1, 1):
            moved = lg - sgn * dlg
            moved[:, c] += 2 * sgn * dlg[:, c]
            z = (moved - moved.max(axis=1, keepdims=True)).astype(f32)
            e = (np.exp(z.astype(np.float64)) * (1 + sgn * gr.EX2_REL)).astype(f32)
            s = e.sum(axis=1, dtype=f32)
            got = (e[:, c] * (f32(1) / s)).astype(np.float64)
            assert (np.abs(got - p[:, c]) <= dp[:, c]).all(), c


def test_ulp16():
    assert gr.ulp16(1.0) == 2.0 ** -10
    assert gr.ulp16(0.75) == 2.0 ** -11
    assert gr.ulp16(1e-6) == 2.0 ** -24
