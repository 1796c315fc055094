"""Float64 reference of one step of each recurrent back end, with a rounding bound for every output element.

Each step models the operand roundings the kernel applies and nothing else; every other source of
difference is in the bound, derived from the kernel's arithmetic:

- accumulation: the deterministic worst case of any summation order in fp32, (terms) * 2^-24 * sum|terms|
  (no order or internal precision is assumed for the tcgen05 accumulator);
- activations: ex2.approx.ftz / rcp.approx.ftz at their PTX ISA accuracy plus the roundings of the
  shared-reciprocal helpers (gru_tc.cu: recip4_1p_exp2), or expf / tanhf / IEEE division at their CUDA
  accuracy (gru.cu, gru_octbit.cu: the build has no fast-math);
- everything propagated through h' = u h + (1 - u) c, the FC and the softmax.

Tensor-core kernel (gru_tc.cu, api.cu):
- weights: fp16 hi, and lo = RN16(w - hi) for a split layer 0 (pack_tc_weights);
- layer-0 x: tc::split_half8, hi = RN16(x), lo = RN16(x - hi); unsplit: hi only (tc_pack_x_kernel);
- h and r*h: RN16 (tc::pack_half2); the layer above reads RN16(h') (the fp16 hand-off);
- FC: h' = hi + lo and W = hi + lo, two accumulators D[c] = h_hi W_hi + h_lo W_hi and
  D[8 + c] = h_hi W_lo + h_lo W_lo, logits = (D[c] + D[8 + c]) + b.

The octbit step uses oracle/octbit.py, which matches the op bit for bit, and reports per stream whether an
element of [x | r*h] lies close enough to a u8 rounding boundary that the kernel's sigmoid could flip a code.
"""
from __future__ import annotations

import numpy as np

from oracle import model as om
from oracle import octbit as ooct

U = 2.0 ** -24                 # fp32 unit round-off
EX2_REL = 2.0 ** -22           # ex2.approx.ftz.f32: maximum relative error (PTX ISA)
RCP_REL = 2.0 ** -23           # rcp.approx.ftz.f32: 1 ulp (PTX ISA)
EXPF_REL = 2.0 ** -22          # expf, tanhf: 2 ulp (CUDA C++ Programming Guide, single-precision functions)
CLAMP_ABS = 2.0 ** -31 * (1 + 2.0 ** -18)   # recip4_1p_exp2 clamps the exponent at 31: an activation below 2^-31 is
                                            # returned as 1/(1 + 2^31), with the reciprocal's own error
SAFETY = 1.01                  # second-order terms of the first-order propagation below
f16 = np.float16
f32 = np.float32


def rn16(a):
    """Round to fp16 and back, as float64 (numpy rounds to nearest even, subnormals included)."""
    return np.asarray(a, np.float64).astype(f16).astype(np.float64)


def split16(a):
    """x = hi + lo as tc::split_half8 / pack_tc_weights form it from fp32 values."""
    a = np.asarray(a, f32)
    hi = a.astype(f16)
    lo = (a - hi.astype(f32)).astype(f32).astype(f16)
    return hi.astype(np.float64), lo.astype(np.float64)


def ulp16(a):
    """fp16 ulp at |a| (subnormal spacing 2^-24 below 2^-14)."""
    e = np.floor(np.log2(np.maximum(np.abs(a), 2.0 ** -14)))
    return 2.0 ** (e - 10)


def accum_bound(nterms, abs_sum):
    """Worst case of fp32 summation of `nterms` exact products, any order."""
    return nterms * U * abs_sum


def sigmoid(z):
    return 1.0 / (1.0 + np.exp(-z))


# ---------------------------------------------------------------- activation bounds
def tc_act_bound(a, b, dacc, mul):
    """|kernel - exact| of 1 / (1 + 2^(mul (a + b))) as recip4_1p_exp2 evaluates it (gru_tc.cu), where the kernel
    reads the accumulator a with an error of at most `dacc`, b is the bias (pre-scaled by fp32 mul on the host)
    and mul is -log2(e) (sigmoid) or 2 log2(e) (tanh).  Returns (value, bound) in float64.

    e = fma(a, mul32, fl(b mul32)): ln2 |de| <= k (dacc + u (|a| + 2 |b| + |a + b|)), k = |mul| / log2(e).
    d = 1 + ex2(e): relative error (1 - s) (ex2 + ln2 |de|) + u.
    1/d from the shared reciprocal: the other three d cancel exactly (their rounded values appear above and
    below), leaving the roundings of d0 d2, d1 d3, their product, rcp, r (d1 d3) and that times d2: 5u + rcp."""
    k = abs(mul) / np.log2(np.e)
    z = a + b
    e = mul * z
    s = 1.0 / (1.0 + np.exp2(np.clip(e, -1000.0, 1000.0)))
    dz = k * (dacc + U * (np.abs(a) + 2.0 * np.abs(b) + np.abs(z)))
    rel = (1.0 - s) * (EX2_REL + dz) + 6.0 * U + RCP_REL
    bound = s * rel * SAFETY + np.where(e > 30.0, CLAMP_ABS, 0.0)
    return s, bound


def tc_sigmoid(a, b, dacc):
    return tc_act_bound(a, b, dacc, -np.log2(np.e))


def tc_tanh(a, b, dacc):
    s, bs = tc_act_bound(a, b, dacc, 2.0 * np.log2(np.e))
    c = 1.0 - 2.0 * s
    return c, 2.0 * bs + U * np.abs(c) * SAFETY


def f32_sigmoid(a, b, dacc):
    """1 / (1 + expf(-fl(a + b))) with IEEE division (gru.cu: sigmoid_f; gru_octbit.cu)."""
    z = a + b
    s = sigmoid(z)
    dz = dacc + U * np.abs(z)
    return s, s * ((1.0 - s) * (EXPF_REL + dz) + 2.0 * U) * SAFETY


def f32_tanh(a, b, dacc):
    """tanhf(fl(a + b))."""
    c = np.tanh(a + b)
    dz = dacc + U * np.abs(a + b)
    return c, ((1.0 - c * c) * dz + (EXPF_REL + U) * np.abs(c)) * SAFETY


def update_bound(u, du, h, c, dc, fused):
    """h' = u h + (1 - u) c and its bound.  fused (gru_tc.cu): fma(u, fma(c, -1, h), c), two roundings;
    otherwise (gru.cu, gru_octbit.cu) u*h + (1-u)*c with up to four roundings (contracted or not)."""
    hn = u * h + (1.0 - u) * c
    d = du * np.abs(h - c) + np.abs(1.0 - u) * dc
    if fused:
        d = d + U * (np.abs(u * (h - c)) + np.abs(hn))
    else:
        d = d + 4.0 * U * (np.abs(u * h) + np.abs((1.0 - u) * c))
    return hn, d * SAFETY


# ---------------------------------------------------------------- one layer step
def _x_operands(x, split):
    if split:
        return split16(x)
    return rn16(x), None


def tc_layer_step(x, h, gk, gb, ck, cb, split):
    """One tensor-core GRU step of a layer.  x [S, in] fp32 as the kernel receives it (layer 0: the mel; above:
    the layer below's fp32 state, which the kernel reads as RN16), h [S, 128] fp32.  -> (h', bound) float64."""
    x = np.asarray(x, f32)
    h = np.asarray(h, f32).astype(np.float64)
    H = h.shape[1]
    ind = x.shape[1]
    xh, xl = _x_operands(x, split)
    h16 = rn16(h)

    def xpart(W):
        Wx = np.asarray(W[:ind], f32)
        if split:
            Wh_, Wl_ = split16(Wx)
            val = xh @ Wh_ + xl @ Wh_ + xh @ Wl_
            mag = np.abs(xh) @ np.abs(Wh_) + np.abs(xl) @ np.abs(Wh_) + np.abs(xh) @ np.abs(Wl_)
            return val, mag, 3 * ind
        W16 = rn16(Wx)
        return xh @ W16, np.abs(xh) @ np.abs(W16), ind

    gx, gmag, gn = xpart(gk)
    Whg = rn16(np.asarray(gk[ind:], f32))
    ga = gx + h16 @ Whg
    gacc = accum_bound(gn + H, gmag + np.abs(h16) @ np.abs(Whg))
    gb = np.asarray(gb, f32).astype(np.float64)
    r, dr = tc_sigmoid(ga[:, :H], gb[:H], gacc[:, :H])
    u, du = tc_sigmoid(ga[:, H:], gb[H:], gacc[:, H:])
    rh = rn16(r * h)
    drh = np.abs(h) * dr + U * np.abs(r * h) + ulp16(np.abs(r * h) + np.abs(h) * dr)   # one fp16 ulp: the kernel's r is not r
    cx, cmag, cn = xpart(ck)
    Whc = rn16(np.asarray(ck[ind:], f32))
    ca = cx + rh @ Whc
    cacc = accum_bound(cn + H, cmag + (np.abs(rh) + drh) @ np.abs(Whc)) + drh @ np.abs(Whc)
    c, dc = tc_tanh(ca, np.asarray(cb, f32).astype(np.float64), cacc)
    return update_bound(u, du, h, c, dc, fused=True)


def f32_layer_step(x, h, gk, gb, ck, cb):
    """One step of gru.cu's exact-fp32 layer: sequential fmaf over [x | h] rows, expf / tanhf / IEEE division."""
    x = np.asarray(x, f32).astype(np.float64)
    h = np.asarray(h, f32).astype(np.float64)
    H = h.shape[1]
    gk = np.asarray(gk, f32).astype(np.float64)
    ck = np.asarray(ck, f32).astype(np.float64)
    xh = np.concatenate([x, h], axis=1)
    K = xh.shape[1]
    ga = xh @ gk
    gacc = accum_bound(K, np.abs(xh) @ np.abs(gk))
    gb = np.asarray(gb, f32).astype(np.float64)
    r, dr = f32_sigmoid(ga[:, :H], gb[:H], gacc[:, :H])
    u, du = f32_sigmoid(ga[:, H:], gb[H:], gacc[:, H:])
    rh = r * h
    drh = np.abs(h) * dr + U * np.abs(rh)
    xrh = np.concatenate([x, rh], axis=1)
    dx = np.concatenate([np.zeros_like(x), drh], axis=1)
    ca = xrh @ ck
    cacc = accum_bound(K, (np.abs(xrh) + dx) @ np.abs(ck)) + dx @ np.abs(ck)
    c, dc = f32_tanh(ca, np.asarray(cb, f32).astype(np.float64), cacc)
    return update_bound(u, du, h, c, dc, fused=False)


def _quant_codes(v, bscale, offset):
    """The op's u8 code of float64 values for a given fp32 bscale (before the fp32 division's rounding)."""
    return ooct._round_half_away(v / np.float64(bscale)) + offset


def octbit_layer_step(x, h, gk, gb, ck, cb, gmat, cmat):
    """One step of gru_octbit_layer_kernel for each stream (its own op calls: ranges are per stream).
    gmat / cmat: (wq [B, K] int8, scale, obias) as the model holds them.  -> (h', bound, flagged [S] bool,
    quantum [S, 128]: what one u8 code step of each element that could flip adds to |h' - ref|)."""
    x = np.asarray(x, f32)
    h32 = np.asarray(h, f32)
    S, H = h32.shape
    hn = np.zeros((S, H))
    bound = np.zeros((S, H))
    flagged = np.zeros(S, bool)
    quantum = np.zeros((S, H))
    gb = np.asarray(gb, f32)
    cb = np.asarray(cb, f32)
    wqc = np.asarray(cmat[0], np.int64)
    for s in range(S):
        xh = np.concatenate([x[s], h32[s]])[None, :]
        g = ooct.octbit_mat_mul(xh, gmat[0], scale=f32(gmat[1]), bias=gmat[2])[0].astype(np.float64)
        r, dr = f32_sigmoid(g[:H], gb[:H].astype(np.float64), 0.0)
        u, du = f32_sigmoid(g[H:], gb[H:].astype(np.float64), 0.0)
        # the kernel's r*h: fl(r_kernel * h); the reference quantises fl(fl(r) * h) and bounds the difference
        rh32 = (r.astype(f32) * h32[s]).astype(f32)
        drh = np.abs(h32[s]) * (dr + U * r) + 2.0 * U * np.abs(rh32.astype(np.float64))
        xrh = np.concatenate([x[s], rh32])[None, :]
        cpre = ooct.octbit_mat_mul(xrh, cmat[0], scale=f32(cmat[1]), bias=cmat[2])[0].astype(np.float64)
        # which codes the kernel's r*h could change: value and (through the range) bscale both perturbed
        v = xrh[0].astype(np.float64)
        dv = np.concatenate([np.zeros(x.shape[1]), drh])
        _, bscale, signed = ooct.quantize_activations(xrh)
        lo_v, hi_v = v - dv, v + dv
        # the range element: bscale is the reference's exactly unless the largest magnitude can move
        if signed:
            m_hi, m_lo, div = np.max(np.maximum(-lo_v, hi_v)), np.max(np.maximum(-hi_v, lo_v)), 127.0
        else:
            m_hi, m_lo, div = np.max(hi_v), np.max(lo_v), 254.0
        moved = m_hi != m_lo
        b_hi = m_hi / div * (1.0 + 2.0 * U) if moved else np.float64(bscale)
        b_lo = m_lo / div * (1.0 - 2.0 * U) if moved else np.float64(bscale)
        ratios = np.stack([lo_v / b_hi, lo_v / b_lo, hi_v / b_hi, hi_v / b_lo])
        rmin = ratios.min(axis=0)
        rmax = ratios.max(axis=0)
        rmin = rmin - 2.0 * U * np.abs(rmin)                      # the kernel's fp32 division
        rmax = rmax + 2.0 * U * np.abs(rmax)
        may_flip = ((dv > 0) | moved) & (ooct._round_half_away(rmin) != ooct._round_half_away(rmax))
        # a moved range also rescales the op's output (scale * bscale)
        dscale = np.abs(cpre) * ((b_hi - b_lo) / b_lo + 2.0 * U) if moved else 0.0
        c, dc = f32_tanh(cpre, cb.astype(np.float64), dscale)
        hn[s], bound[s] = update_bound(u, du, h32[s].astype(np.float64), c, dc, fused=False)
        if may_flip.any():
            flagged[s] = True
            step = np.float64(cmat[1]) * np.float64(bscale)
            quantum[s] = np.abs(1.0 - u) * (np.abs(wqc[:, may_flip]).sum(axis=1) * step) * SAFETY
    return hn, bound, flagged, quantum


# ---------------------------------------------------------------- FC + softmax
def softmax_bound(lg, dlg, ex_rel, div_rel):
    """softmax(lg) in float64 and a bound for the kernel's: logits off by at most dlg, each exponential of
    (lg - max) with relative error ex_rel + 3u |lg - max| (fl subtraction, fp32 log2(e), fl product), the
    sum's (C - 1) roundings, then the reciprocal/division and product (div_rel)."""
    lg = np.asarray(lg, np.float64)
    z = lg - lg.max(axis=-1, keepdims=True)
    e = np.exp(z)
    p = e / e.sum(axis=-1, keepdims=True)
    C = lg.shape[-1]
    rel_e = ex_rel + 3.0 * U * np.abs(z)
    dl = np.max(dlg, axis=-1, keepdims=True)
    rel = np.expm1(2.0 * dl) + rel_e + rel_e.max(axis=-1, keepdims=True) + (C - 1) * U + div_rel
    return p, (p * rel + 2.0 ** -125) * SAFETY


def tc_fc(h, fc_w, fc_b):
    """FC + softmax of the tensor-core kernel's last layer on its fp32 state h [S, 128]."""
    hh, hl = split16(h)
    Wh, Wl = split16(np.asarray(fc_w, f32))
    d0 = hh @ Wh + hl @ Wh
    d1 = hh @ Wl + hl @ Wl
    b = np.asarray(fc_b, f32).astype(np.float64)
    lg = d0 + d1 + b
    K = 2 * h.shape[1]
    dlg = (accum_bound(K, np.abs(hh) @ np.abs(Wh) + np.abs(hl) @ np.abs(Wh)) +
           accum_bound(K, np.abs(hh) @ np.abs(Wl) + np.abs(hl) @ np.abs(Wl)) +
           U * np.abs(d0 + d1) + U * np.abs(lg)) * SAFETY
    p, dp = softmax_bound(lg, dlg, EX2_REL, RCP_REL + U)
    return lg, dlg, p, dp


def f32_fc(h, fc_w, fc_b):
    """FC + softmax of gru.cu's last layer (and of the octbit graph's float FC): fmaf over the 128 units from 0,
    + b, expf, IEEE division."""
    h = np.asarray(h, f32).astype(np.float64)
    W = np.asarray(fc_w, f32).astype(np.float64)
    lg = h @ W + np.asarray(fc_b, f32).astype(np.float64)
    dlg = (accum_bound(h.shape[1], np.abs(h) @ np.abs(W)) + U * np.abs(lg)) * SAFETY
    p, dp = softmax_bound(lg, dlg, EXPF_REL, U)
    return lg, dlg, p, dp


def octbit_fc_logits(y, fc_mat, fc_b):
    """Logits of fc_octbit_softmax_kernel for one stream's frames y [n, 128]: one op call over the frames, + b
    in fp32.  Bit for bit what the kernel computes."""
    lg = ooct.octbit_mat_mul(np.asarray(y, f32), fc_mat[0], scale=f32(fc_mat[1]), bias=fc_mat[2])
    return (lg + np.asarray(fc_b, f32)).astype(f32)


# ---------------------------------------------------------------- layer-0 plan of the tensor-core kernel
def tc_plan(n_mel: int, num_layers: int, cap: int):
    """(split, x buffers) of layer 0; 0 buffers: the model runs the fp32 kernel (api.cu: tc_fits)."""
    return om.tc_layer0_plan(n_mel, num_layers, cap)


def tc_regime(n_mel: int, num_layers: int, cap: int) -> str:
    split, nbuf = tc_plan(n_mel, num_layers, cap)
    if nbuf == 0:
        return "fp32"
    return "%s%d" % ("split" if split else "unsplit", nbuf)
