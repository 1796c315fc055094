"""GPU: the attention_ctc kernels one at a time against float64 references, and the whole forward pass at the
configurations kws_attention_create accepts.

The model-level tests in test_gpu_attention.py see each kernel only through layer norms over whole utterances and a
softmax over the classes, which flatten most errors of a single kernel.  Here every kernel runs alone on inputs built
to expose its own edges (kws_debug_att_*), and every element is held to an error bound derived from the kernel's
arithmetic instead of one flat tolerance.
"""
import math
from dataclasses import dataclass

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                     # fp32 unit roundoff
LOG2E = 1.4426950408889634
HEAD = 16                          # head size the attention kernels are built for
TC, FFMA = 0, 1                    # the `path` argument of the debug entry points
KWS_ERR_UNSUPPORTED = -4


def _lib():
    from keyword_spotting_b200 import _lib as lib_mod
    return lib_mod, lib_mod.load()


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def _f64(a):
    import torch
    return torch.from_numpy(np.asarray(a, np.float64)).cuda()


# ================================================================ dense layers
# Y[r, n] = act(sum_k A[r, k] W[k, n] + bias[n]) (+ pe[r % Tp, n]).  Let M[r, n] = (|A| |W|)[r, n] + |bias[n]| (+ |pe|).
#
# FFMA (att_linear_kernel): K fmaf roundings into one fp32 accumulator, each at most u times the partial sum of
#   |a_k w_k| <= M, then one rounding each for + bias and + pe; relu is exact and 1-Lipschitz:  |err| <= (K + 2) u M.
#
# tcgen05 (att_linear_tc_kernel): x = hi + lo with hi = fp16(x), lo = fp16(x - hi); x - hi is exact in fp32 and
#   |x - hi| <= 2^-11 |x|, so |x - hi - lo| <= 2^-22 |x|, or <= 2^-25 absolute when lo falls in fp16's subnormal range
#   (|x| below about 2^-3 .. 2^-14).  The kernel sums  A_hi W_hi + A_lo W_hi + A_hi W_lo:  the splits of a and w cost
#   2^-22 each and the dropped A_lo W_lo another 2^-22 (times |a w|), i.e. 3 * 2^-22 M, plus the absolute part
#   2^-25 (1 + 2^-10) (sum_k |W[k, n]| + sum_k |A[r, k]|) < 2^-24 (colsum |W| + rowsum |A|).  fp16 x fp16 products are
#   exact in fp32; each of the 3 ceil(K / 16) MMAs adds its sum into the fp32 accumulator with at most one rounding
#   of 2^-23 M (2^-23, not 2^-24, so that a hardware that truncates is covered as well); + bias and + pe add 2 u M.
def eps_ffma_linear(K):
    return (K + 2) * U


def eps_tc_linear(K):
    return 3 * 2.0 ** -22 + 3 * math.ceil(K / 16) * 2.0 ** -23 + 2 * U


def _dense_inputs(rng, rows, K, N, Tp):
    """Rows at scales from 1e-4 to 3e3 (log-uniform), a few all-zero rows, mostly negative biases (relu clips them),
    a few weights 300 times larger than the rest.  |values| stay far below fp16's 65520 (see kws_b200.h)."""
    A = rng.standard_normal((rows, K)) * np.exp(rng.uniform(math.log(1e-4), math.log(3e3), rows))[:, None]
    if rows > 2:
        A[rng.random(rows) < 0.03] = 0.0
        A[rows // 2] = 0.0
    W = rng.standard_normal((K, N)) / math.sqrt(K)
    big = rng.choice(K * N, min(8, K * N), replace=False)
    W.flat[big] *= 300.0
    bias = rng.standard_normal(N) - 0.7
    pe = rng.standard_normal((Tp, N))
    return A.astype(np.float32), W.astype(np.float32), bias.astype(np.float32), pe.astype(np.float32)


def _dense_reference(A, W, bias, pe, Tp, relu, add_pe):
    """float64 value, the magnitude M and the absolute term of the tcgen05 bound (all [rows, N], on the device)."""
    import torch
    A64, W64, b64 = _f64(A), _f64(W), _f64(bias)
    want = A64 @ W64 + b64
    mag = A64.abs() @ W64.abs() + b64.abs()
    if relu:
        want = want.clamp_min(0.0)
    if add_pe:
        pr = _f64(pe)[torch.arange(A.shape[0], device="cuda") % Tp]
        want, mag = want + pr, mag + pr.abs()
    absterm = 2.0 ** -24 * (A64.abs().sum(1, keepdim=True) + W64.abs().sum(0, keepdim=True))
    return want, mag, absterm


def _run_linear(A_d, W, bias_d, pe_d, Tp, rows, K, N, relu, add_pe, path):
    import torch
    lib_mod, lib = _lib()
    Y = torch.full((rows, N), float("nan"), dtype=torch.float32, device="cuda")
    rc = lib.kws_debug_att_linear(A_d.data_ptr(), np.ascontiguousarray(W).ctypes.data, bias_d.data_ptr(),
                                  pe_d.data_ptr(), Tp, rows, K, N, int(relu), int(add_pe), path, Y.data_ptr(), _stream())
    return rc, Y, lib_mod


def _tc_supported(K, N):
    return N % 128 == 0 and K % 4 == 0


# (K, N, rows, relu, add_pe, Tp): every K with the tile edge rows = 129, every N and every variant at 4133 rows (T' = 51 and
# 400 put r % T' boundaries inside and across the 128-row tiles), every row count at an N of three column tiles.
_DENSE_CASES = sorted(
    {(K, 128, 129, True, True, 51) for K in (4, 60, 64, 68, 120, 128, 200, 512, 1024)}
    | {(120, N, 4133, False, True, 400) for N in (128, 384, 512, 1024)}
    | {(68, 384, rows, True, False, 51) for rows in (1, 100, 128, 129, 4133)}
    | {(128, 512, 4133, relu, pe, Tp) for relu in (False, True) for pe in (False, True) for Tp in (51, 400)}
    | {(1024, 1024, 4133, True, True, 400), (200, 128, 4133, False, False, 400), (4, 1024, 100, False, True, 51)}
    # the FFMA kernel alone: N not a multiple of 128 (6 = the class count), K not a multiple of 4
    | {(120, N, 4133, True, True, 400) for N in (6, 64, 65, 200, 512)}
    | {(K, N, rows, True, True, 51) for K in (41, 82, 123) for N, rows in ((128, 4133), (65, 129), (200, 1))}
    | {(K, 64, 4133, False, False, 400) for K in (4, 60, 200, 512, 1024)})


def _check_linear(K, N, rows, relu, add_pe, Tp):
    """Both kernels (the tensor cores where they take the shape) against float64; returns err / bound per path."""
    rng = np.random.default_rng(K * 7919 + N * 31 + rows + 2 * relu + add_pe + Tp)
    A, W, bias, pe = _dense_inputs(rng, rows, K, N, Tp)
    A_d, bias_d, pe_d = _dev(A), _dev(bias), _dev(pe)
    want, mag, absterm = _dense_reference(A, W, bias, pe, Tp, relu, add_pe)
    got = {}
    for path, eps, extra in ((FFMA, eps_ffma_linear(K), 0.0), (TC, eps_tc_linear(K), absterm)):
        rc, Y, lib_mod = _run_linear(A_d, W, bias_d, pe_d, Tp, rows, K, N, relu, add_pe, path)
        if path == TC and not _tc_supported(K, N):
            assert rc == KWS_ERR_UNSUPPORTED
            continue
        lib_mod.check(rc)
        bound = eps * mag + extra
        err = (Y.double() - want).abs()
        worst = float((err / bound).max())
        assert worst <= 1.0, ("path", path, "err/bound", worst, "max err", float(err.max()))
        got[path] = (Y.double(), bound, worst)
    if len(got) == 2:                          # the two kernels agree within the sum of their bounds
        (y0, b0, _), (y1, b1, _) = got[TC], got[FFMA]
        assert float(((y0 - y1).abs() / (b0 + b1)).max()) <= 1.0
    return {p: g[2] for p, g in got.items()}


@pytest.mark.parametrize("K,N,rows,relu,add_pe,Tp", _DENSE_CASES)
def test_att_linear_matches_float64(K, N, rows, relu, add_pe, Tp):
    _check_linear(K, N, rows, relu, add_pe, Tp)


def test_att_linear_rejects_shapes_the_tensor_cores_do_not_take():
    import torch
    lib_mod, lib = _lib()
    A = torch.zeros((4, 64), device="cuda")
    Y = torch.zeros((4, 200), device="cuda")
    b = torch.zeros(200, device="cuda")
    W = np.zeros((64, 200), np.float32)
    assert lib.kws_debug_att_linear(A.data_ptr(), W.ctypes.data, b.data_ptr(), None, 1, 4, 64, 200, 0, 0, TC,
                                    Y.data_ptr(), _stream()) == KWS_ERR_UNSUPPORTED
    assert "N % 128" in lib_mod.last_error()
    assert lib.kws_debug_att_linear(A.data_ptr(), W.ctypes.data, b.data_ptr(), None, 1, 4, 62, 128, 0, 0, TC,
                                    Y.data_ptr(), _stream()) == KWS_ERR_UNSUPPORTED


# ================================================================ attention core
# Per (utterance b, head h): o_i = sum_j p_ij v_j / sum_j p_ij with p_ij = 2^(s_ij - max_j s_ij), s = q k^T / 4 in log2
# units.  If every p_ij carries a relative error of at most d_p, then |o~_i - o_i| <= d_p / (1 - d_p) sum_j P_ij |v_j - o_i|
# (P the exact softmax); errors in the products p v and their accumulation add e_v sum_j P_ij |v_j|.  A score error of
# at most e_s A_i, A_i = max_j sum_d |q_id k_jd| / 4 log2(e), moves p_ij by ln 2 (|ds_ij| + |ds_max|) <= 2 ln 2 e_s A_i:
#     |err_id| <= (2 ln 2 e_s A_i + e_p) sum_j P_ij |v_jd - o_id| + e_v sum_j P_ij |v_jd| + a_id
#
# tcgen05 (att_core_tc_kernel): scores from hi/lo splits of q (after the fp32 scaling) and k, three MMAs:
#   e_s = 3 * 2^-22 + 3 * 2^-23 + u.  p: ex2.approx (relative error < 2^-22), the hi/lo split of p (2^-22) and the
#   row sum, sequential over at most ceil(T' / 32) * 16 keys per thread and then one add:  e_p = 2^-21 + (T' / 2 + 18) u.
#   p v: hi/lo splits of p and v (2 * 2^-22, the dropped lo x lo 2^-22), 3 MMAs per 16 keys into fp32 (2^-23 each,
#   truncation-safe) and the final scaling:  e_v = 3 * 2^-22 + 3 ceil(T' / 16) 2^-23 + 2u.  a: a lo part in fp16's
#   subnormal range is off by up to 2^-25 absolute; for v that adds 2^-25 sum_j P_ij = 2^-25, for a p below 2^-14
#   2^-25 |v_jd| / sum_j p_ij:  a_id = 2^-25 (1 + sum_{j: p_ij < 2^-14} |v_jd| / sum_j p_ij).
# FFMA (att_attention_kernel): 16 fmaf after the fp32 scaling of q:  e_s = 18u.  exp2f (2 ulp) and up to T' rescales of
#   the running sum and output when the maximum moves:  e_p = 3 (T' + 4) u.  T' fmaf into o:  e_v = (T' + 4) u;  a = 0.
@dataclass
class CoreEps:
    s: float
    p: float
    v: float
    subnormal_lo: bool


def eps_tc_core(Tp):
    return CoreEps(3 * 2.0 ** -22 + 3 * 2.0 ** -23 + U, 2.0 ** -21 + (Tp / 2 + 18) * U,
                   3 * 2.0 ** -22 + 3 * math.ceil(Tp / 16) * 2.0 ** -23 + 2 * U, True)


def eps_ffma_core(Tp):
    return CoreEps(18 * U, 3 * (Tp + 4) * U, (Tp + 4) * U, False)


def _split_qkv(qkv, heads):
    """[B, T', 3 * 16 * heads] -> q, k, v as [B, heads, T', 16] float64 (device)."""
    x = _f64(qkv)
    B, Tp, _ = x.shape
    return [x[:, :, i * heads * HEAD:(i + 1) * heads * HEAD].reshape(B, Tp, heads, HEAD).transpose(1, 2)
            for i in range(3)]


def _core_reference(qkv, heads):
    """float64 output [B, T', 16 heads] and the per-element pieces of the bound above."""
    import torch
    q, k, v = _split_qkv(qkv, heads)
    s = q @ k.transpose(-1, -2) * (0.25 * LOG2E)                          # log2 units
    P = torch.softmax(s * math.log(2.0), dim=-1)
    o = P @ v
    A = ((q.abs() @ k.abs().transpose(-1, -2)) * (0.25 * LOG2E)).amax(-1, keepdim=True)
    spread = torch.stack([(P * (v[..., d].unsqueeze(2) - o[..., d].unsqueeze(3)).abs()).sum(-1) for d in range(HEAD)], -1)
    absv = P @ v.abs()
    small = (s - s.amax(-1, keepdim=True)) < -14.0                        # p < 2^-14: lo part of p subnormal
    sub = 2.0 ** -25 * (small.double() @ v.abs()) * P.amax(-1, keepdim=True)   # 1 / sum_j p_ij = max_j P_ij
    return o, A, spread, absv, sub


def _flat(t):
    B, H, Tp, D = t.shape
    return t.transpose(1, 2).reshape(B, Tp, H * D)


def _core_bound(ref, eps):
    o, A, spread, absv, sub = ref
    b = (2 * math.log(2.0) * eps.s * A + eps.p) * spread + eps.v * absv
    if eps.subnormal_lo:
        b = b + sub + 2.0 ** -25
    return _flat(b)


def _run_core(qkv_d, B, Tp, heads, path):
    import torch
    lib_mod, lib = _lib()
    out = torch.full((B, Tp, heads * HEAD), float("nan"), dtype=torch.float32, device="cuda")
    rc = lib.kws_debug_att_core(qkv_d.data_ptr(), B, Tp, heads, path, out.data_ptr(), _stream())
    return rc, out, lib_mod


_GOOD_KEY_COS = 0.85


def _unit(rng, shape):
    x = rng.standard_normal(shape)
    return x / np.linalg.norm(x, axis=-1, keepdims=True)


def _core_inputs(kind, rng, B, Tp, heads):
    """qkv [B, T', 3 * 16 * heads] fp32 and, for 'peaked', the key planted for each query [B, heads, T'].
      generic  Gaussian q, k, v
      peaked   every query has one dominant key (score >= 30 log2 units above every other): keys 0 and T' - 1, a key of
               the padded last group, both sides of the g_split boundary between the two warps of a lane quarter and
               keys 255 / 256 (the second score MMA) for chosen queries, random keys for the rest
      equal    q = 0: all scores equal, o = mean(v), which pins the padded-key masks
      spread   scores spread over +-60 log2 units
      offset   Gaussian q, k and a distinct offset of v per (b, h), so that mixing up heads or utterances shows
    peaked and equal carry the per-(b, h) v offsets as well."""
    N = heads * HEAD
    q = rng.standard_normal((B, heads, Tp, HEAD))
    k = rng.standard_normal((B, heads, Tp, HEAD))
    v = rng.standard_normal((B, heads, Tp, HEAD))
    offs = 4.0 * (np.arange(B * heads).reshape(B, heads, 1, 1) + 1) * np.where(np.arange(heads) % 2, -1, 1)[None, :, None, None]
    target = None
    if kind in ("peaked", "equal", "offset"):
        v = v + offs
    if kind == "equal":
        q[:] = 0.0
    elif kind == "spread":
        s = np.einsum("bhid,bhjd->bhij", q, k) * 0.25 * LOG2E
        q *= 60.0 / np.abs(s).max()
    elif kind == "peaked":
        k = _unit(rng, (B, heads, Tp, HEAD))
        groups = (Tp + 15) // 16
        g_split = (groups + 1) // 2
        special_keys = [0, Tp - 1, 16 * (groups - 1), 16 * g_split - 1, 16 * g_split, 255, 256]
        special_keys = sorted({j for j in special_keys if 0 <= j < Tp})
        special_rows = sorted({i for i in (0, 31, 32, 63, 64, 95, 96, 127, 128, 255, 256, 383, 384, Tp - 1) if i < Tp})
        target = rng.integers(0, Tp, (B, heads, Tp))
        for n, i in enumerate(special_rows):
            target[:, :, i] = special_keys[n % len(special_keys)]
        for b in range(B):
            for h in range(heads):
                kk = k[b, h]
                for j in special_keys:                         # re-draw a planted special key until it stands apart
                    others = np.delete(kk, j, axis=0)
                    while others.size and (others @ kk[j]).max() > _GOOD_KEY_COS:
                        kk[j] = _unit(rng, HEAD)
                cos = kk @ kk.T
                np.fill_diagonal(cos, -1.0)
                closest = cos.max(1)
                good = np.flatnonzero(closest <= _GOOD_KEY_COS)
                t = target[b, h]
                bad = ~np.isin(t, special_keys) & (closest[t] > _GOOD_KEY_COS)
                t[bad] = good[rng.integers(0, len(good), int(bad.sum()))]
                # q = beta k_t: the planted key scores beta / 4 log2(e), key j beta cos(t, j) / 4 log2(e), 33 less at most
                gap = 1.0 - np.maximum(closest[t], 0.0)
                beta = 33.0 / (0.25 * LOG2E * gap)
                q[b, h] = beta[:, None] * kk[t]
    qkv = np.concatenate([x.transpose(0, 2, 1, 3).reshape(B, Tp, N) for x in (q, k, v)], axis=2)
    return qkv.astype(np.float32), target


def _check_core(kind, Tp, path, heads=8, B=2, seed=0, also_ffma=False):
    rng = np.random.default_rng(seed * 100003 + Tp * 7 + path)
    qkv, target = _core_inputs(kind, rng, B, Tp, heads)
    qkv_d = _dev(qkv)
    ref = _core_reference(qkv, heads)
    want = _flat(ref[0])
    results = {}
    for p in ((TC, FFMA) if also_ffma else (path,)):
        rc, out, lib_mod = _run_core(qkv_d, B, Tp, heads, p)
        lib_mod.check(rc)
        bound = _core_bound(ref, eps_tc_core(Tp) if p == TC else eps_ffma_core(Tp))
        err = (out.double() - want).abs()
        worst = float((err / bound).max())
        assert worst <= 1.0, (kind, "T'", Tp, "path", p, "err/bound", worst, "max err", float(err.max()))
        results[p] = (out.double(), bound, worst)
        if kind == "peaked":                       # the output is the planted key's v, so a row or key mix-up is O(1)
            import torch
            _, _, v = _split_qkv(qkv, heads)
            t = torch.from_numpy(target).cuda()
            vt = torch.gather(v, 2, t.unsqueeze(-1).expand(-1, -1, -1, HEAD))
            dv = float((out.double() - _flat(vt)).abs().max())
            assert dv < 1e-5, (kind, "T'", Tp, "path", p, "|o - v_planted|", dv)
        if kind == "equal":
            _, _, v = _split_qkv(qkv, heads)
            mean = _flat(v.mean(2, keepdim=True).expand(-1, -1, Tp, -1))
            assert float((out.double() - mean).abs().max()) < 1e-5 * float(mean.abs().max() + 1)
    if also_ffma:
        (y0, b0, _), (y1, b1, _) = results[TC], results[FFMA]
        assert float(((y0 - y1).abs() / (b0 + b1)).max()) <= 1.0, ("tc vs ffma", kind, Tp)
    return {p: r[2] for p, r in results.items()}


_KINDS = ("generic", "peaked", "equal", "spread", "offset")


@pytest.mark.parametrize("kind", _KINDS)
def test_att_core_tc_every_key_count(kind):
    """Every T' the tensor-core core takes: T' % 16 (the padded last key group), 1..4 live lane quarters of the last
    query tile, odd and even key-group counts (g_split) and the second score MMA from key 256 on.  generic and spread
    also run the FFMA core on the same inputs and hold the two against each other."""
    for Tp in range(1, 401):
        _check_core(kind, Tp, TC, also_ffma=kind in ("generic", "spread"))


@pytest.mark.parametrize("kind", _KINDS)
@pytest.mark.parametrize("Tp", [1, 127, 128, 129, 400, 401, 513, 1000])
def test_att_core_ffma_matches_float64(kind, Tp):
    _check_core(kind, Tp, FFMA, seed=1)


def test_att_core_tc_rejects_more_than_400_keys():
    import torch
    lib_mod, lib = _lib()
    qkv = torch.zeros((1, 401, 384), device="cuda")
    out = torch.zeros((1, 401, 128), device="cuda")
    assert lib.kws_debug_att_core(qkv.data_ptr(), 1, 401, 8, TC, out.data_ptr(), _stream()) == KWS_ERR_UNSUPPORTED


# ================================================================ add + layer norm
# y = (x - mean) / sqrt(var + 1e-12) * gamma + beta over one utterance's n = T' N values, x = a + b in fp32.
#   x: one rounding, |dx| <= u |x|.  mean: each of the 1024 threads sums m = ceil(n / 4096) float4 pieces (2 roundings
#   inside a piece, m - 1 into its partial sum), then 10 levels of shuffle / shared-memory tree:  |dmean| <= (m + 12) u
#   mean|x|.  var: the same sum of squares of x - mean:  relative (m + 14) u, plus 2 mean|x - mean| (u max|x| + dmean)
#   absolute.  1 / sqrt: relative dvar / (2 var) + 2u.  Output:
#     |err| <= |g| inv (u |x| + dmean) + |g| |x - mean| inv (dinv + 3u) + u |y|
def _ln_reference(a, b, gamma, beta, Tp, N):
    x = _f64(a) + _f64(b)
    B = x.shape[0]
    x = x.reshape(B, Tp * N)
    mean = x.mean(1, keepdim=True)
    d = x - mean
    var = (d * d).mean(1, keepdim=True)
    inv = 1.0 / (var + 1e-12).sqrt()
    g, be = _f64(gamma).repeat(Tp), _f64(beta).repeat(Tp)
    y = d * inv * g + be
    m = math.ceil(Tp * N / 4096)
    dmean = (m + 12) * U * x.abs().mean(1, keepdim=True)
    dvar = (m + 14) * U * var + 2 * d.abs().mean(1, keepdim=True) * (U * x.abs().amax(1, keepdim=True) + dmean)
    dinv = dvar / (2 * var) + 2 * U
    bound = g.abs() * inv * (U * x.abs() + dmean) + g.abs() * d.abs() * inv * (dinv + 3 * U) + U * y.abs()
    return y.reshape(B, Tp, N), bound.reshape(B, Tp, N)


def _check_layernorm(Tp, in_smem):
    import torch
    lib_mod, lib = _lib()
    B, N = 3, 128
    rng = np.random.default_rng(Tp * 2 + in_smem)
    a = (1e3 + rng.standard_normal((B, Tp, N))).astype(np.float32)
    b = rng.standard_normal((B, Tp, N)).astype(np.float32)
    gamma = (1 + 0.3 * rng.standard_normal(N)).astype(np.float32)
    beta = rng.standard_normal(N).astype(np.float32)
    a_d, b_d, g_d, be_d = _dev(a), _dev(b), _dev(gamma), _dev(beta)
    y = torch.full((B, Tp, N), float("nan"), device="cuda")
    rc = lib.kws_debug_att_add_layernorm(a_d.data_ptr(), b_d.data_ptr(), g_d.data_ptr(), be_d.data_ptr(), B, Tp, N,
                                         in_smem, y.data_ptr(), _stream())
    if in_smem and Tp * N * 4 > 200 * 1024:
        assert rc == KWS_ERR_UNSUPPORTED
        return 0.0
    lib_mod.check(rc)
    want, bound = _ln_reference(a, b, gamma, beta, Tp, N)
    err = (y.double() - want).abs()
    worst = float((err / bound).max())
    assert worst <= 1.0, (worst, float(err.max()))
    return worst


@pytest.mark.parametrize("Tp", [1, 400, 401])
@pytest.mark.parametrize("in_smem", [1, 0])
def test_att_add_layernorm_matches_float64(Tp, in_smem):
    """A large common offset (1e3) on unit-variance data: a one-pass E[x^2] - E[x]^2 would lose the variance."""
    _check_layernorm(Tp, in_smem)


# ================================================================ the model at other configurations
# combine_frame == 1 is left out: kws_attention_frames gives T' = T there, the oracle's padding rule gives T + 1, and
# without the reference's source nothing here settles which one the reference computes.
def _model(n_mel=60, combine=2, layers=3, ffn=512, classes=6, relu=True, seed=4321):
    from keyword_spotting_b200 import AttentionConfig, AttentionDeployModel, AttentionWeights
    from oracle import attention as oa

    @dataclass
    class Config(AttentionConfig):
        classes: int = 6

        @property
        def num_classes(self):
            return self.classes

    ow = oa.init_weights(seed=seed, n_mel=n_mel, combine=combine, layers=layers, ffn=ffn, classes=classes)
    cfg = Config(n_mel=n_mel, combine_frame=combine, num_layers=layers, feed_forward_inner_size=ffn, use_relu=relu,
                 classes=classes)
    return ow, AttentionDeployModel(cfg, AttentionWeights.from_object(ow))


def _check_model(ow, m, B, T, seed):
    from oracle import attention as oa
    c = m.config
    rng = np.random.default_rng(seed)
    mel = (np.abs(rng.standard_normal((B, T, c.n_mel))) * rng.uniform(0.2, 3.0)).astype(np.float32)
    want, lwant = oa.mel_forward(mel, ow, np.float32, use_relu=c.use_relu, combine=c.combine_frame)
    want64, _ = oa.mel_forward(mel, ow, np.float64, use_relu=c.use_relu, combine=c.combine_frame)
    got, lgot = m.run_mel(mel, want_logits=True)
    assert got.shape == want.shape == (B, T // c.combine_frame + 1, c.num_classes)
    assert np.abs(got - want64).max() < 1e-3, np.abs(got - want64).max()
    assert np.abs(got - want).max() < 1e-4, np.abs(got - want).max()
    assert np.abs(lgot - lwant).max() < 1e-3
    return mel, got


# (n_mel, combine, layers, ffn, classes, relu).  ffn = 200: ff1 on the FFMA kernel (N % 128 != 0), ff2 on the tensor
# cores with K = 200.  n_mel = 41, combine = 3: K = 123, the input layer on the FFMA kernel, and B T' odd (3 x 33) puts
# every scratch segment after the first at an odd float offset unless the forward pads them.
_CONFIGS = [(40, 2, 3, 512, 6, True), (60, 3, 3, 512, 6, True), (60, 2, 3, 256, 6, True), (60, 2, 3, 200, 6, True),
            (60, 2, 3, 1024, 6, True), (60, 2, 1, 512, 6, True), (60, 2, 8, 512, 6, True), (60, 2, 3, 512, 2, True),
            (60, 2, 3, 512, 16, True), (60, 2, 3, 512, 6, False), (41, 3, 3, 512, 6, True)]


@pytest.mark.parametrize("n_mel,combine,layers,ffn,classes,relu", _CONFIGS)
def test_attention_config_matches_oracle(n_mel, combine, layers, ffn, classes, relu):
    ow, m = _model(n_mel, combine, layers, ffn, classes, relu, seed=n_mel + 10 * layers + ffn + classes)
    try:
        T_odd = 33 * combine - 1 if combine > 1 else 33          # T' = 33
        _check_model(ow, m, 3, T_odd, seed=1)
        _check_model(ow, m, 2, 799, seed=2)
    finally:
        m.close()


@pytest.fixture(scope="module")
def default_model():
    ow, m = _model()
    yield ow, m
    m.close()


@pytest.mark.parametrize("T", [799, 800])
def test_attention_at_the_tensor_core_limit(default_model, T):
    """T' = 400 and 401: the attention core moves from tcgen05 to FFMA and the layer norm from shared to global memory."""
    ow, m = default_model
    _check_model(ow, m, 3, T, seed=T)


def test_attention_chunks_across_max_rows_per_call(default_model):
    ow, m = default_model
    mel, whole = _check_model(ow, m, 7, 100, seed=11)           # T' = 51
    m.MAX_ROWS_PER_CALL = 3 * 51 + 7                            # 3 utterances per call: 3 + 3 + 1
    try:
        chunked = m.run_mel(mel)
    finally:
        del m.MAX_ROWS_PER_CALL
    np.testing.assert_array_equal(chunked, whole)


def test_attention_scratch_and_pe_regrow_and_shrink(default_model):
    """A sequence of calls that grows and shrinks B and T re-allocates the scratch and the positional encoding; every
    result equals that of a model that has seen no other call."""
    from keyword_spotting_b200 import AttentionDeployModel, AttentionWeights
    ow, _ = default_model
    m = AttentionDeployModel(default_model[1].config, AttentionWeights.from_object(ow))
    try:
        rng = np.random.default_rng(3)
        for B, T in [(2, 100), (5, 799), (1, 40), (9, 300), (2, 1000), (3, 61), (1, 799)]:
            mel = np.abs(rng.standard_normal((B, T, 60))).astype(np.float32)
            got = m.run_mel(mel)
            fresh = AttentionDeployModel(m.config, AttentionWeights.from_object(ow))
            try:
                np.testing.assert_array_equal(got, fresh.run_mel(mel))
            finally:
                fresh.close()
    finally:
        m.close()
