// K2+K3 on the 5th-generation tensor cores: persistent recurrent GRU (TF GRUCell semantics) + FC + softmax.
//
// Same maths as gru.cu (models/rnn_ctc.py:156-165,202-284; reset gate applied BEFORE the candidate matmul):
//   [r,u] = sigmoid([x,h] Wg + bg),  c = tanh([x, r*h] Wc + bc),  h' = u*h + (1-u)*c,  softmax(h' Wfc + bfc)
//
// Mapping to sm_100a:
//   * one CTA owns 128 streams for a whole layer -- the streams are the M dimension of tcgen05.mma
//     (M=128, cta_group::1); the TMEM lane of a stream is owned by the same thread for the whole chunk, so the
//     fp32 master state h never leaves registers between time steps;
//   * all weights of the layer ([384, K] fp16, 172-196 KB) are resident in shared memory for the whole
//     kernel, in the K-major SWIZZLE_NONE canonical layout, packed on the host at model creation;
//   * the recurrent A operand (h_{t-1}, then r*h) lives in TENSOR MEMORY (TS-form MMA): each thread writes its own
//     stream's row with tcgen05.st, so the recurrent activations never touch shared memory;
//   * the input A operand x_t never touches a thread at all: the producer of x (the front end for layer 0, the
//     layer below otherwise) leaves it in HBM as fp16 in the row-tiled operand layout (tc05.cuh: [tile][t][K/8 chunks]
//     [128 streams][8 elements]), so ONE bulk async copy (cp.async.bulk, completion on an mbarrier) per tile-step
//     lands an MMA-ready SS-form operand in shared memory, double-buffered, a step ahead;
//   * TMEM map (512 columns): D_r 0..127, D_u 128..255, D_cand 256..383, A_h 384..447;
//   * the input projection is not a separate GEMM: x_t W[0:in] is accumulated into the same TMEM tile as
//     h W[in:], and it is issued a phase early so it never sits on the recurrent critical path;
//   * warp-specialised: warps 0-15 run the gate algebra from TMEM (warp w: the 32 streams of TMEM lane quarter w%4,
//     hidden units [32*(w/4), +32) -- four warps per scheduler hide the MUFU / TMEM-load latencies); warp 16 issues
//     the bulk copies and the MMAs.  Everything is handed over with mbarriers (tcgen05.commit and copy completion one
//     way, 512-thread arrivals the other) -- no CTA-wide barrier inside the time loop.  Per step:
//         warp 16                                          gate threads
//         r-gate h-part -> commit R      <- A_h ready      ...
//         copy x_{t+1} -> other buffer
//         u-gate x+h    -> commit U                        wait R: r = sigmoid(D_r), keep fp16(r*h) in registers
//         cand  x-part                                     wait U: A_h <- r*h, arrive;  u = sigmoid(D_u) -> registers
//         cand  h-part  -> commit C      <- A_rh ready     wait C: c = tanh(D_c), h' = c + u (h - c), A_h <- h', arrive
//         r-gate x-part of step t+1      <- x_{t+1} landed FC partials / softmax / hand-off stores of step t
//     so the dependent chain of a step is  r-MMA(h) -> sigmoid -> cand-MMA(h) -> tanh,  with the u gate, all
//     x-part MMAs, the copies, the softmax and the global stores running beside it;
//   * gate algebra in fp32 with ex2.approx / rcp.approx and packed f32x2 arithmetic (FFMA2/FADD2/FMUL2); activations
//     are evaluated four at a time sharing one reciprocal (5 MUFU per 4 activations, 3.75 per hidden unit and step),
//     biases pre-scaled by log2(e).  Each accumulator column is read from TMEM exactly once per step (the TMEM read
//     port moves 64 B/clk: a [128,128] fp32 gate costs 1024 cycles per read).
// Operands are fp16 (weights rounded once on the host, activations rounded by their producer), accumulation
// and all state fp32.  The layer-0 input projection is the exception: mel features are unbounded (tens for loud
// audio) and a single fp16 rounding of x and W_x alone costs up to 3e-3 on the carried state, so that product is
// issued as three fp16 MMAs  x_hi*W_hi + x_lo*W_hi + x_hi*W_lo  (x = x_hi + x_lo, W = W_hi + W_lo; the
// dropped lo*lo term is 2^-22 relative), i.e. at fp32-grade accuracy for +6 small MMAs per step: the front end
// writes both halves of the split.  With it the deviation from the fp32 graph stays below 1e-3 (contract) on
// probabilities and state; see DESIGN.md.
#include <type_traits>
#include <vector>

#include "common.cuh"
#include "tc05.cuh"

namespace kws {

constexpr int kTcTile = 128;
constexpr int kTcEpiWarps = 16;           // warps 0-15: gate algebra.  Warp w owns TMEM lanes 32*(w%4).. (its 32 streams)
constexpr int kTcEpiThreads = 32 * kTcEpiWarps;   //   and the 32 hidden units [32*(w/4), +32) of those streams
constexpr int kTcThreads = kTcEpiThreads + 128;   // + warpgroup 4: warp 16 issues the x copies and the MMAs (warps 17-19 only donate registers)
constexpr int kTcUnits = 32;              // hidden units per gate thread
constexpr int kFcOperandBytes = 16 * kHidden * 2;   // FC weights as an MMA operand: N = 16 (8 classes, hi and lo), K = 128


struct GruTcParams {
  int kx;                      // x width padded to a multiple of 16
  int kxw;                     // x columns of the operand and of the packed weights: 2*kx when the x product is split
  int nbuf;                    // x buffers in shared memory: 2, or 1 when two do not fit
  long S;
  int n;                       // frames of the whole sequence: the time stride of x, the hand-off, probs and logits
  int t0, nt;                  // this launch runs frames [t0, t0 + nt) (the layers of long sequences are pipelined in time chunks)
  const unsigned char* x_tiles;   // layer 0: fp16 row-tiled operand [tile][t][kxw/8 chunks][128 streams][8]: [x_hi | x_lo (split)]
  const __half* x_f16;         // layers above: the layer below's outputs, same layout with 16 chunks
  __half* y_f16;               // non-last layers: outputs in that layout
  const __half* wpack;         // [384, kxw+128] fp16, canonical layout: [Wx_hi | Wx_lo (split only) | Wh]
  const float* bias;           // [384] = gates (r | u) | candidate
  const float* h_in;           // [S, 128]
  float* h_out;                // [S, 128]
  const int* seq_len;
  const unsigned char* zero_state;
  int C;
  float* probs;                // [S, n, C]
  float* logits;               // [S, n, C] or null
  // FC weights [128][8] + bias [8] by value (copied to shared memory by the last layer's CTAs)
  float fcw[kHidden * kTcMaxClasses];
  float fcb[kTcMaxClasses];
};

constexpr float kLog2e = 1.4426950408889634f;

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// sigmoid(a + b) with nb = -log2(e) * b:   1 / (1 + 2^(-log2e*(a+b)))         FFMA, EX2, FADD, RCP
__device__ __forceinline__ float sigmoid_pre(float a, float nb) {
  return rcp_approx(1.0f + ex2_approx(fmaf(a, -kLog2e, nb)));
}
// tanh(a + b) with pb = 2*log2(e) * b:     1 - 2 / (1 + 2^(2*log2e*(a+b)))    FFMA, EX2, FADD, RCP, FFMA
__device__ __forceinline__ float tanh_pre(float a, float pb) {
  return fmaf(-2.0f, rcp_approx(1.0f + ex2_approx(fmaf(a, 2.0f * kLog2e, pb))), 1.0f);
}

// Two activations for three MUFU operations: 1/d0 and 1/d1 from ONE reciprocal of d0*d1.  The exponents are
// clamped to 63 so that the product stays finite (d <= 2^63 + 1; sigmoid below 1e-19 / tanh above 1 - 2e-19 are
// returned exactly as the clamp leaves them -- far below fp32 resolution of the results).
__device__ __forceinline__ void sigmoid2_pre(float a0, float nb0, float a1, float nb1, float& s0, float& s1) {
  const float d0 = 1.0f + ex2_approx(fminf(fmaf(a0, -kLog2e, nb0), 63.0f));
  const float d1 = 1.0f + ex2_approx(fminf(fmaf(a1, -kLog2e, nb1), 63.0f));
  const float r = rcp_approx(d0 * d1);
  s0 = r * d1;
  s1 = r * d0;
}
__device__ __forceinline__ void tanh2_pre(float a0, float pb0, float a1, float pb1, float& c0, float& c1) {
  const float d0 = 1.0f + ex2_approx(fminf(fmaf(a0, 2.0f * kLog2e, pb0), 63.0f));
  const float d1 = 1.0f + ex2_approx(fminf(fmaf(a1, 2.0f * kLog2e, pb1), 63.0f));
  const float r = rcp_approx(d0 * d1);
  c0 = fmaf(-2.0f, r * d1, 1.0f);
  c1 = fmaf(-2.0f, r * d0, 1.0f);
}

// Four activations for FIVE MUFU operations and packed f32x2 arithmetic: with d = 1 + 2^e, the four reciprocals
// come from ONE reciprocal of d0*d1*d2*d3:  P = (d0 d2, d1 d3),  r = 1/(P.x P.y),  Rinv = r (P.y, P.x) = (1/(d0 d2),
// 1/(d1 d3)),  (1/d0, 1/d1) = Rinv (d2, d3),  (1/d2, 1/d3) = Rinv (d0, d1).  The exponents are clamped to 31 so that the
// product stays finite (<= 2^124); a sigmoid below 5e-10 / a tanh above 1 - 1e-9 is returned as the clamp leaves it.
// Inputs: a = accumulator values, b = bias pre-scaled by `mul` (the activation is act(a + bias)), mul = -log2(e) for
// the sigmoid and 2 log2(e) for tanh.  Output: 1 / (1 + 2^(mul * (a + bias))) for the four inputs.
__device__ __forceinline__ void recip4_1p_exp2(float2 a01, float2 a23, float2 b01, float2 b23, float mul,
                                               float2& s01, float2& s23) {
  const float2 m2 = make_float2(mul, mul);
  float2 e01 = __ffma2_rn(a01, m2, b01), e23 = __ffma2_rn(a23, m2, b23);
  e01.x = ex2_approx(fminf(e01.x, 31.0f));
  e01.y = ex2_approx(fminf(e01.y, 31.0f));
  e23.x = ex2_approx(fminf(e23.x, 31.0f));
  e23.y = ex2_approx(fminf(e23.y, 31.0f));
  const float2 one = make_float2(1.0f, 1.0f);
  const float2 d01 = __fadd2_rn(e01, one), d23 = __fadd2_rn(e23, one);
  const float2 pp = __fmul2_rn(d01, d23);
  const float r = rcp_approx(pp.x * pp.y);
  const float2 rinv = __fmul2_rn(make_float2(r, r), make_float2(pp.y, pp.x));
  s01 = __fmul2_rn(rinv, d23);
  s23 = __fmul2_rn(rinv, d01);
}
__device__ __forceinline__ void sigmoid4_pre(float2 a01, float2 a23, float2 nb01, float2 nb23, float2& s01, float2& s23) {
  recip4_1p_exp2(a01, a23, nb01, nb23, -kLog2e, s01, s23);
}
__device__ __forceinline__ void tanh4_pre(float2 a01, float2 a23, float2 pb01, float2 pb23, float2& c01, float2& c23) {
  float2 s01, s23;
  recip4_1p_exp2(a01, a23, pb01, pb23, 2.0f * kLog2e, s01, s23);
  const float2 m2 = make_float2(-2.0f, -2.0f), one = make_float2(1.0f, 1.0f);
  c01 = __ffma2_rn(s01, m2, one);
  c23 = __ffma2_rn(s23, m2, one);
}
__device__ __forceinline__ float2 u2f2(uint32_t a, uint32_t b) { return make_float2(__uint_as_float(a), __uint_as_float(b)); }

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
// this thread's TMEM stores are complete and ordered before the arrival
__device__ __forceinline__ void tmem_publish(uint64_t* bar) {
  tc::wait_st();
  tc::fence_before_sync();
  mbar_arrive(bar);
}
__device__ __forceinline__ void mbar_acquire(uint64_t* bar, uint32_t parity) {
  tc::mbar_wait(bar, parity);
  tc::fence_after_sync();
}

enum { kBarXF0 = 0, kBarXF1, kBarAX, kBarXD, kBarAH, kBarARH, kBarR, kBarU, kBarC, kBarF, kBarFR, kNumBars };

// kXSmem: the x operand arrives in shared memory by bulk copy (layer 0: 24 KB per tile-step next to 172 KB of weights).
//   The layers above (32 KB per tile-step next to 196 KB of weights: no room) take x through the gate threads into
//   TMEM columns 448..511 instead, loaded a step ahead.
// kNX: k16 steps of the x operand when they are known at compile time, so that the issuing warp runs straight-line
//   code -- 8: a 128-wide layer below (not split), 3: the 40-mel front end (split); 0: taken from the parameters.
template <bool kLast, bool kXSmem, int kNX>
__global__ void __launch_bounds__(kTcThreads, 1)
gru_tc_kernel(const GruTcParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int ktot = p.kxw + kHidden;                                                  // K extent of the packed weights
  const uint32_t xbytes = static_cast<uint32_t>(p.kxw / 8) * tc::kTileChunkBytes;    // one tile-step of x
  unsigned char* sW = smem;                                                         // [384, ktot] fp16
  unsigned char* sX = sW + static_cast<size_t>(768) * ktot;                         // kXSmem: [nbuf][kxw/8 chunks][128][8] fp16
  float* sBias = reinterpret_cast<float*>(sX + (kXSmem ? static_cast<size_t>(p.nbuf) * xbytes : 0));   // [384] pre-scaled
  unsigned char* sWfc = reinterpret_cast<unsigned char*>(sBias + 384);     // [16, 128] fp16 canonical: FC weights, rows 0-7 hi, 8-15 lo (last layer)
  float* sProb = reinterpret_cast<float*>(sWfc + kFcOperandBytes);         // [4 steps][6][128] parked probabilities (last layer)
  float* sLg = sProb + 4 * 6 * kTcTile;                                    // [8][128] logits between their read and the softmax (last layer)
  uint64_t* bars = reinterpret_cast<uint64_t*>(kLast ? sLg + kTcMaxClasses * kTcTile : sBias + 384);   // [kNumBars]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kNumBars);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int kMmaWarp = kTcEpiWarps;

  if (warp == kMmaWarp) tc::tmem_alloc(tmem_slot, 512);
  if (tid == 0) {
    tc::mbar_init(&bars[kBarXF0], 1);               // the issuing lane's arrive.expect_tx + the copy's bytes
    tc::mbar_init(&bars[kBarXF1], 1);
    tc::mbar_init(&bars[kBarAX], kTcEpiThreads);
    tc::mbar_init(&bars[kBarXD], 1);
    tc::mbar_init(&bars[kBarAH], kTcEpiThreads);
    tc::mbar_init(&bars[kBarARH], kTcEpiThreads);
    tc::mbar_init(&bars[kBarR], 1);
    tc::mbar_init(&bars[kBarU], 1);
    tc::mbar_init(&bars[kBarC], 1);
    tc::mbar_init(&bars[kBarF], 1);
    tc::mbar_init(&bars[kBarFR], kTcTile);          // the 128 threads of unit block 0 read the logits
    tc::mbar_fence_init();
  }
  {
    const int n16 = 384 * ktot * 2 / 16;
    const uint4* src = reinterpret_cast<const uint4*>(p.wpack);
    for (int i = tid; i < n16; i += kTcThreads) reinterpret_cast<uint4*>(sW)[i] = __ldg(src + i);
    for (int i = tid; i < 384; i += kTcThreads)
      sBias[i] = p.bias[i] * (i < 2 * kHidden ? -kLog2e : 2.0f * kLog2e);
    if (kLast)                                       // B operand of the FC: row c = fp16(W[:, c]), row 8 + c = what that rounding lost
      for (int i = tid; i < 16 * kHidden; i += kTcThreads) {
        const int n = i >> 7, k = i & (kHidden - 1);
        const float w = p.fcw[k * kTcMaxClasses + (n & 7)];
        const __half hi = __float2half_rn(w);
        *reinterpret_cast<__half*>(sWfc + tc::canon_offset(n, k, kHidden)) = n < 8 ? hi : __float2half_rn(w - __half2float(hi));
      }
  }
  tc::fence_proxy_async();            // weights written with generic stores, read by the MMA (async proxy)
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();

  const uint32_t tmem = *tmem_slot;
  const uint32_t colDr = 0, colDu = 128, colDc = 256, colAh = 384, colAx = 448;
  const long ntiles = (p.S + kTcTile - 1) / kTcTile;
  const int t_end = p.t0 + p.nt;

  if (warp >= kMmaWarp) {
    // =========================================================== x copies + MMA issue (one elected lane of warp 16)
    // (setmaxnreg is a warpgroup-wide instruction: warps 16-19 must all execute the same one)
    asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
    if (warp == kMmaWarp) {
    const int nx = kNX ? kNX : p.kx / 16;
    const bool split = kNX ? kNX == 3 : p.kxw != p.kx;             // 3-term x product
    const bool two = p.nbuf == 2;
    const uint32_t sbo = static_cast<uint32_t>(ktot / 8) * 128;
    const uint32_t idesc128 = tc::idesc_f16(128, 128);
    // All operand addresses are computed warp-uniformly (they live in uniform registers); the MMAs of a group are issued
    // from ONE elect.sync region (tc::elect_one): back-to-back UTCHMMA, no per-instruction lane loop.  B descriptor of K-chunk k16 for the weight rows starting at row0 =
    // base + ((row0/8)*sbo + 256*k16)/16 added to the 14-bit start-address field (shared memory < 256 KB: no carry).
    const uint64_t wbase = tc::smem_desc(tc::smem_u32(sW), 128, sbo);
    const uint32_t row_step = (16 * sbo) >> 4;                             // 128 output rows
    const uint64_t xdesc0 = tc::smem_desc(tc::smem_u32(sX), tc::kTileChunkBytes, 128);   // A, row-tiled: LBO 2048 (K), SBO 128 (M)
    const uint64_t xdesc1 = xdesc0 + (xbytes >> 4);
    constexpr uint32_t kStepA = (2 * tc::kTileChunkBytes) >> 4;           // one k16 step of the A operand: two chunks
    // The TMEM base comes out of shared memory, i.e. in a vector register the compiler cannot prove warp-uniform: every
    // TMEM operand address derived from it would be hoisted out of the time loop as an invariant and, at 32 registers,
    // spilled to local memory and reloaded per MMA.  `tm` is redefined (opaquely) at every step, so the addresses are
    // recomputed next to their MMA instead: one add in the uniform datapath.
    uint32_t tm = tmem;
    uint64_t wb = wbase, xd0 = xdesc0, xd1 = xdesc1;       // (same for the descriptor bases: 64-bit invariants per gate and K step otherwise)
    // x-part of a product into D columns `dcol` (overwrites D), weight rows starting at 128*rblk
    auto issue_x_from = [&](uint64_t xdesc, uint32_t dcol, int rblk) {
      const uint64_t wrow = wb + rblk * row_step;
      const uint64_t xlo = xdesc + static_cast<uint64_t>(nx) * kStepA;    // the lo chunks follow the hi chunks
      if (tc::elect_one()) {
#pragma unroll
        for (int k16 = 0; k16 < (kNX ? kNX : nx); ++k16)                   // x_hi * Wx_hi
          tc::mma_ss(tm + dcol, xdesc + k16 * kStepA, wrow + 16 * k16, idesc128, k16 > 0);
        if (split) {
#pragma unroll
          for (int k16 = 0; k16 < (kNX ? kNX : nx); ++k16)                 // x_lo * Wx_hi
            tc::mma_ss(tm + dcol, xlo + k16 * kStepA, wrow + 16 * k16, idesc128, true);
#pragma unroll
          for (int k16 = 0; k16 < (kNX ? kNX : nx); ++k16)                 // x_hi * Wx_lo
            tc::mma_ss(tm + dcol, xdesc + k16 * kStepA, wrow + 16 * (nx + k16), idesc128, true);
        }
      }
    };
    // (the buffer index is loop-carried, which the compiler cannot prove warp-uniform: branch on it so that every
    // descriptor is derived from kernel constants and stays in uniform registers)
    auto issue_x = [&](int buf, uint32_t dcol, int rblk) {
      if (!kXSmem) {                                                       // x in TMEM (never split: a layer's outputs are in [-1, 1])
        const uint64_t wrow = wb + rblk * row_step;
        if (tc::elect_one()) {
#pragma unroll
          for (int k16 = 0; k16 < (kNX ? kNX : nx); ++k16)
            tc::mma_ts(tm + dcol, tm + colAx + 8 * k16, wrow + 16 * k16, idesc128, k16 > 0);
        }
      } else if (buf == 0) {
        issue_x_from(xd0, dcol, rblk);
      } else {
        issue_x_from(xd1, dcol, rblk);
      }
    };
    const int nxw = p.kxw / 16;
    auto issue_h = [&](uint32_t dcol, int rblk) {                          // += A_h * Wh[128*rblk .. +127]
      const uint64_t wrow = wb + rblk * row_step + 16 * nxw;
      if (tc::elect_one()) {
#pragma unroll
        for (int k16 = 0; k16 < kHidden / 16; ++k16)
          tc::mma_ts(tm + dcol, tm + colAh + 8 * k16, wrow + 16 * k16, idesc128, true);
      }
    };
    auto prefetch = [&](long tile, int t, int buf) {                       // x of (tile, t) -> buffer `buf`
      if (tc::elect_one()) {
        tc::mbar_arrive_expect_tx(&bars[kBarXF0 + buf], xbytes);
        tc::bulk_g2s(sX + static_cast<size_t>(buf) * xbytes, p.x_tiles + (tile * p.n + t) * static_cast<long>(xbytes), xbytes,
                     &bars[kBarXF0 + buf]);
      }
    };
    // FC on the tensor core (last layer): logits(t) = h'(t) Wfc with h' = hi + lo (two fp16 terms, exact to 2^-22) and
    // Wfc = hi + lo packed as the 16 rows of one N = 16 operand: D_fc[c] + D_fc[8 + c].  A_hi is A_h (the next step's
    // recurrent operand anyway); A_lo is parked by the gate threads in the columns of D_u they own (free between the
    // u gate's read and the next u-gate MMAs, which are issued behind these); D_fc borrows candidate columns 0..15
    // (free until the next candidate x-part, which waits for the logits to be read: kBarFR).
    const uint32_t idesc16 = tc::idesc_f16(128, 16);
    const uint64_t fdesc = tc::smem_desc(tc::smem_u32(sWfc), 128, (kHidden / 8) * 128);
    uint64_t fd = fdesc;
    auto issue_fc = [&]() {
      if (tc::elect_one()) {
#pragma unroll
        for (int j = 0; j < kHidden / 16; ++j) tc::mma_ts(tm + colDc, tm + colAh + 8 * j, fd + 16 * j, idesc16, j > 0);
#pragma unroll
        for (int j = 0; j < kHidden / 16; ++j)
          tc::mma_ts(tm + colDc, tm + colDu + 32 * (j >> 1) + 8 * (j & 1), fd + 16 * j, idesc16, true);
        tc::commit(&bars[kBarF]);
      }
    };
    uint32_t it = 0;                                                       // (tile, step) pairs done by this CTA
    uint32_t ah = 0, nf = 0;                                               // A_h hand-overs consumed, FC products issued
    if (static_cast<long>(blockIdx.x) < ntiles && p.nt > 0) {
      if (kXSmem) {
        prefetch(blockIdx.x, p.t0, 0);
        mbar_acquire(&bars[kBarXF0], 0);
      } else {
        mbar_acquire(&bars[kBarAX], 0);
      }
      issue_x(0, colDr, 0);                                                // r gate, x-part of the very first step
    }
    for (long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      for (int t = p.t0; t < t_end; ++t, ++it) {
        const uint32_t par = it & 1;
        const int buf = two ? static_cast<int>(it & 1) : 0;
        asm volatile("" : "+r"(tm), "+l"(wb), "+l"(xd0), "+l"(xd1), "+l"(fd));
        const bool step_next = t + 1 < t_end;
        const long ntile = step_next ? tile : tile + gridDim.x;            // what this CTA runs next
        const int nt1 = step_next ? t + 1 : p.t0;
        const bool has_next = ntile < ntiles;
        mbar_acquire(&bars[kBarAH], ah & 1);                               // h_{t-1} in A_h; every MMA of the previous step is complete
        ++ah;
        issue_h(colDr, 0);
        if (tc::elect_one()) tc::commit(&bars[kBarR]);
        if (kLast && t > p.t0) {                                           // logits of the previous step, behind the critical r gate
          issue_fc();
          ++nf;
        }
        if (kXSmem && two && has_next) prefetch(ntile, nt1, buf ^ 1);      // the other buffer's last readers were the previous step's MMAs
        issue_x(buf, colDu, 1);                                            // u gate
        issue_h(colDu, 1);
        if (tc::elect_one()) tc::commit(&bars[kBarU]);
        if (kLast && nf > 0) mbar_acquire(&bars[kBarFR], (nf - 1) & 1);    // the logits have left the candidate columns
        issue_x(buf, colDc, 2);                                            // candidate, x-part
        if (!kXSmem && tc::elect_one()) tc::commit(&bars[kBarXD]);                    // A_x has been read: the gate threads may store x_{t+1}
        mbar_acquire(&bars[kBarARH], par);                                 // r*h in A_h (and D_r read by every gate thread)
        issue_h(colDc, 2);
        if (tc::elect_one()) tc::commit(&bars[kBarC]);
        if (kLast && !step_next) {                                         // the tile's last step: its logits are not followed by an r gate
          mbar_acquire(&bars[kBarAH], ah & 1);
          ++ah;
          issue_fc();
          ++nf;
        }
        if (has_next) {
          if (kXSmem) {
            int nb = buf ^ 1;
            uint32_t xpar = ((it + 1) >> 1) & 1;
            if (!two) {                                                    // one buffer: it is free once this step's MMAs are complete
              mbar_acquire(&bars[kBarC], par);
              prefetch(ntile, nt1, 0);
              nb = 0;
              xpar = (it + 1) & 1;
            }
            mbar_acquire(&bars[kBarXF0 + nb], xpar);
            issue_x(nb, colDr, 0);                                         // next r gate, x-part: queued behind this step's candidate
          } else {
            mbar_acquire(&bars[kBarAX], par ^ 1);
            issue_x(0, colDr, 0);
          }
        }
      }
    }
    }
  } else {
    // =========================================================== gate algebra (512 threads: one stream x 32 units each)
    asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");      // launched at 96: 128 x (96-32) released = 512 x (112-96) acquired
    const int quarter = warp & 3, ublk = warp >> 2;
    const int row = 32 * quarter + lane;
    const uint32_t lane_sel = static_cast<uint32_t>(32 * quarter) << 16;
    const int u0 = kTcUnits * ublk;                                 // first hidden unit of this thread
    const uint32_t my_ah = tmem + lane_sel + colAh + 16 * ublk;     // 32 units = 16 columns
    const uint32_t my_alo = tmem + lane_sel + colDu + 32 * ublk;    // last layer: fp16(h' - fp16(h')) in the first 16 of this thread's own D_u columns
    uint32_t nf = 0;                                                // FC products consumed
    const float* bR = sBias + u0;
    const float* bU = sBias + kHidden + u0;
    const float* bC = sBias + 2 * kHidden + u0;
    // last layer, the model's 6 classes, 16-byte aligned rows: probabilities leave four steps at a time (fc_finish)
    const bool probs_batched = kLast && p.C == 6 && ((p.n | p.t0) & 1) == 0 && (reinterpret_cast<uintptr_t>(p.probs) & 15) == 0;
    uint32_t it = 0;

    for (long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      const long s = tile * kTcTile + row;
      const bool ok = s < p.S;
      const long sr = ok ? s : 0;
      const int len = ok ? (p.seq_len ? p.seq_len[s] : p.n) : 0;
      const bool all_live = __all_sync(0xffffffffu, len >= t_end);   // warp-uniform: no select in the update
      float h[kTcUnits];
      {
        const bool zero = !ok || (p.zero_state && p.zero_state[s]);
        const float4* src = reinterpret_cast<const float4*>(p.h_in + sr * kHidden + u0);
#pragma unroll
        for (int i = 0; i < kTcUnits / 4; ++i) {
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (!zero) v = src[i];
          h[4 * i] = v.x; h[4 * i + 1] = v.y; h[4 * i + 2] = v.z; h[4 * i + 3] = v.w;
        }
      }
      // layers above the first: x_t of this thread = K elements [32*ublk, +32) of its stream's row, loaded a step ahead
      uint32_t xr[kXSmem ? 1 : 16];
      const uint32_t my_ax = tmem + lane_sel + colAx + 16 * ublk;
      auto load_x = [&](int t) {
        if (!kXSmem) {
          // chunk q of stream `row` sits at ((tile*n + t)*16 + q)*128 + row: a warp reads 512 contiguous bytes
          const uint4* src = reinterpret_cast<const uint4*>(p.x_f16) + ((tile * p.n + t) * 16 + 4 * ublk) * kTcTile + row;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint4 v = __ldg(src + q * kTcTile);
            xr[kXSmem ? 0 : 4 * q] = v.x; xr[kXSmem ? 0 : 4 * q + 1] = v.y;
            xr[kXSmem ? 0 : 4 * q + 2] = v.z; xr[kXSmem ? 0 : 4 * q + 3] = v.w;
          }
        }
      };
      auto store_x = [&]() {
        if (!kXSmem) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint32_t v[4] = {xr[kXSmem ? 0 : 4 * q], xr[kXSmem ? 0 : 4 * q + 1], xr[kXSmem ? 0 : 4 * q + 2],
                                   xr[kXSmem ? 0 : 4 * q + 3]};
            tc::st4(my_ax + 4 * q, v);
          }
        }
      };
      auto store_h = [&]() {                                       // A_h <- fp16(h)
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          uint32_t v[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = tc::pack_half2(h[16 * c + 2 * i], h[16 * c + 2 * i + 1]);
          tc::st8(my_ah + 8 * c, v);
        }
      };
      // Last layer: the logits of a step come out of the tensor core during the NEXT step (issue_fc above); the 128 threads
      // of unit block 0 read them (16 TMEM columns: hi-weight and lo-weight halves), release the columns and finish
      // softmax + stores in the shadow of the candidate MMAs.  dynamic_rnn: zero output past the length, i.e. logits = bias.
      auto read_logits = [&](uint32_t fpar, bool emit) {
        mbar_acquire(&bars[kBarF], fpar);
        uint32_t v[16];
        tc::ld16(tmem + lane_sel + colDc, v);
        tc::wait_ld();
        tc::fence_before_sync();
        mbar_arrive(&bars[kBarFR]);
#pragma unroll
        for (int c = 0; c < kTcMaxClasses; ++c)          // parked in shared memory (this thread's column): 8 registers less under the r*h hand-over
          sLg[c * kTcTile + row] = (emit ? __uint_as_float(v[c]) + __uint_as_float(v[8 + c]) : 0.0f) + p.fcb[c];
      };
      auto emit_probs = [&](int t_done) {
        if (!ok) return;
        float lg[kTcMaxClasses];
        float mx = -INFINITY;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          lg[c] = sLg[c * kTcTile + row];
          if (c < p.C) mx = fmaxf(mx, lg[c]);
        }
        float e[8], sum = 0.0f;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          e[c] = c < p.C ? ex2_approx((lg[c] - mx) * kLog2e) : 0.0f;    // 2 ulp: far inside the 1e-3 contract
          sum += e[c];
        }
        const float inv = rcp_approx(sum);                              // sum in [1, C]
        if (probs_batched) {
          // Probabilities of four consecutive steps are parked in shared memory (a column per stream, touched by
          // this thread only) and leave as 96 contiguous bytes per stream: 3 full sectors instead of 4 x 24
          // scattered bytes.
          const int kq = (t_done - p.t0) & 3;
#pragma unroll
          for (int c = 0; c < 6; ++c) sProb[(kq * 6 + c) * kTcTile + row] = e[c] * inv;
          if (kq == 3 || t_done == t_end - 1) {
            float4* dst = reinterpret_cast<float4*>(p.probs + (s * p.n + (t_done - kq)) * 6);
            const int nq4 = ((kq + 1) * 6) >> 2;                 // whole float4s: 6 (4 steps), 4, 3, 1
#pragma unroll
            for (int i = 0; i < 6; ++i)
              if (i < nq4)
                dst[i] = make_float4(sProb[(4 * i) * kTcTile + row], sProb[(4 * i + 1) * kTcTile + row],
                                     sProb[(4 * i + 2) * kTcTile + row], sProb[(4 * i + 3) * kTcTile + row]);
            float* tail = reinterpret_cast<float*>(dst) + 4 * nq4;   // (kq+1)*6 mod 4 = 2 left over when kq is 0 or 2
            if (((kq + 1) * 6) & 3) {
              tail[0] = sProb[(4 * nq4) * kTcTile + row];
              tail[1] = sProb[(4 * nq4 + 1) * kTcTile + row];
            }
          }
        } else {
          float* pr = p.probs + (s * p.n + t_done) * p.C;
#pragma unroll
          for (int c = 0; c < 8; ++c)
            if (c < p.C) pr[c] = e[c] * inv;
        }
        if (p.logits) {
          float* lo = p.logits + (s * p.n + t_done) * p.C;
#pragma unroll
          for (int c = 0; c < 8; ++c)
            if (c < p.C) lo[c] = lg[c];
        }
      };
      bool emit_prev = false;                                      // whether the previous step was inside its stream's length

      // ---- prologue: A_h <- fp16(h).  All MMAs of the previous tile have completed (its last commit was waited
      // for by every thread), so the operand region is free.
      if (!kXSmem) {
        load_x(p.t0);
        store_x();
      }
      store_h();
      tc::wait_st();
      tc::fence_before_sync();
      if (!kXSmem) mbar_arrive(&bars[kBarAX]);
      mbar_arrive(&bars[kBarAH]);

      for (int t = p.t0; t < t_end; ++t, ++it) {
        const uint32_t par = it & 1;
        const bool more = t + 1 < t_end;
        if (!kXSmem && more) load_x(t + 1);                        // coalesced global loads in flight under the r gate
        // ---- r gate: keep fp16(r*h) in registers until the u-gate MMAs have finished reading A_h
        uint32_t rh[kTcUnits / 2];
        mbar_acquire(&bars[kBarR], par);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          uint32_t v[16];
          tc::ld16(tmem + lane_sel + colDr + u0 + 16 * c, v);
          tc::wait_ld();
#pragma unroll
          for (int i = 0; i < 16; i += 4) {
            const int j = 16 * c + i;
            const float4 nb = *reinterpret_cast<const float4*>(bR + j);
            float2 r01, r23;
            sigmoid4_pre(u2f2(v[i], v[i + 1]), u2f2(v[i + 2], v[i + 3]), make_float2(nb.x, nb.y), make_float2(nb.z, nb.w), r01, r23);
            const float2 rh01 = __fmul2_rn(r01, make_float2(h[j], h[j + 1]));
            const float2 rh23 = __fmul2_rn(r23, make_float2(h[j + 2], h[j + 3]));
            rh[j / 2] = tc::pack_half2(rh01.x, rh01.y);
            rh[j / 2 + 1] = tc::pack_half2(rh23.x, rh23.y);
          }
        }
        const bool have_logits = kLast && t > p.t0;                // the previous step's, issued behind this step's r gate
        if (have_logits) {
          if (ublk == 0) read_logits(nf & 1, emit_prev);
          ++nf;
        }
        mbar_acquire(&bars[kBarU], par);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const uint32_t v[8] = {rh[8 * c], rh[8 * c + 1], rh[8 * c + 2], rh[8 * c + 3],
                                 rh[8 * c + 4], rh[8 * c + 5], rh[8 * c + 6], rh[8 * c + 7]};
          tc::st8(my_ah + 8 * c, v);
        }
        tmem_publish(&bars[kBarARH]);
        if (have_logits && ublk == 0) emit_probs(t - 1);
        // ---- u gate (beside the candidate MMAs): read once, kept in registers until the update
        float u[kTcUnits];
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          uint32_t v[16];
          tc::ld16(tmem + lane_sel + colDu + u0 + 16 * c, v);
          tc::wait_ld();
#pragma unroll
          for (int i = 0; i < 16; i += 4) {
            const float4 nb = *reinterpret_cast<const float4*>(bU + 16 * c + i);
            float2 u01, u23;
            sigmoid4_pre(u2f2(v[i], v[i + 1]), u2f2(v[i + 2], v[i + 3]), make_float2(nb.x, nb.y), make_float2(nb.z, nb.w), u01, u23);
            u[16 * c + i] = u01.x;
            u[16 * c + i + 1] = u01.y;
            u[16 * c + i + 2] = u23.x;
            u[16 * c + i + 3] = u23.y;
          }
          if (!kXSmem && c == 0 && more) {
            // next step's x: the x-part MMAs of this step were committed right behind the u gate, so A_x is free by now;
            // stored between the halves of the u gate so that x and the whole u are never in registers together
            mbar_acquire(&bars[kBarXD], par);
            store_x();
            tmem_publish(&bars[kBarAX]);
          }
        }
        // ---- candidate and state update: only what the next step's MMAs wait for
        mbar_acquire(&bars[kBarC], par);
        const bool live = t < len;
        // (last layer: 8 units per pass -- with the lo halves of h' the 16-unit pass does not fit the 112 registers, and a
        // spilled loop scalar costs an L2 round trip here: the L1 is 28 KB next to 227 KB of shared memory)
        constexpr int kCw = kLast ? 8 : 16;
#pragma unroll
        for (int c = 0; c < kTcUnits / kCw; ++c) {
          uint32_t vc[kCw];
          if constexpr (kCw == 16) tc::ld16(tmem + lane_sel + colDc + u0 + kCw * c, vc);
          else tc::ld8(tmem + lane_sel + colDc + u0 + kCw * c, vc);
          tc::wait_ld();
          uint32_t packed[kCw / 2];
          uint32_t packed_lo[kLast ? kCw / 2 : 1];
#pragma unroll
          for (int i = 0; i < kCw; i += 4) {
            const int j = kCw * c + i;
            const float4 pb = *reinterpret_cast<const float4*>(bC + j);
            float2 c01, c23;
            tanh4_pre(u2f2(vc[i], vc[i + 1]), u2f2(vc[i + 2], vc[i + 3]), make_float2(pb.x, pb.y), make_float2(pb.z, pb.w), c01, c23);
            const float2 neg = make_float2(-1.0f, -1.0f);
            const float2 h01 = make_float2(h[j], h[j + 1]), h23 = make_float2(h[j + 2], h[j + 3]);
            float2 n01 = __ffma2_rn(make_float2(u[j], u[j + 1]), __ffma2_rn(c01, neg, h01), c01);          // u*h + (1-u)*c
            float2 n23 = __ffma2_rn(make_float2(u[j + 2], u[j + 3]), __ffma2_rn(c23, neg, h23), c23);
            if (!all_live) {                                       // dynamic_rnn: state carried past the length
              n01 = live ? n01 : h01;
              n23 = live ? n23 : h23;
            }
            h[j] = n01.x;
            h[j + 1] = n01.y;
            h[j + 2] = n23.x;
            h[j + 3] = n23.y;
            const __half2 p01 = __floats2half2_rn(n01.x, n01.y), p23 = __floats2half2_rn(n23.x, n23.y);
            packed[i / 2] = *reinterpret_cast<const uint32_t*>(&p01);
            packed[i / 2 + 1] = *reinterpret_cast<const uint32_t*>(&p23);
            if (kLast) {                                           // what the rounding lost: the FC's second operand
              const float2 b01 = __half22float2(p01), b23 = __half22float2(p23);
              packed_lo[kLast ? i / 2 : 0] = tc::pack_half2(n01.x - b01.x, n01.y - b01.y);
              packed_lo[kLast ? i / 2 + 1 : 0] = tc::pack_half2(n23.x - b23.x, n23.y - b23.y);
            }
          }
          if constexpr (kLast) {
            const uint32_t vhi[4] = {packed[0], packed[1], packed[2], packed[3]};
            const uint32_t vlo[4] = {packed_lo[0], packed_lo[kLast ? 1 : 0], packed_lo[kLast ? 2 : 0], packed_lo[kLast ? 3 : 0]};
            tc::st4(my_ah + 4 * c, vhi);
            tc::st4(my_alo + 4 * c, vlo);
          } else {
            if (more) {
              const uint32_t vhi[8] = {packed[0], packed[1], packed[2], packed[3], packed[kLast ? 0 : 4], packed[kLast ? 0 : 5],
                                       packed[kLast ? 0 : 6], packed[kLast ? 0 : 7]};
              tc::st8(my_ah + 8 * c, vhi);
            }
          }
        }
        if (kLast || more) tmem_publish(&bars[kBarAH]);            // releases the next step's r/u MMAs (last layer: and this step's FC)
        // ---- outputs of this step, in the shadow of the next step's r-gate MMAs.  dynamic_rnn: zero output past the length
        const bool emit = all_live || live;
        if (!kLast) {
          // the next layer's x operand, row-tiled (rows past S are written too: the scratch is padded to whole tiles)
          uint4* dst = reinterpret_cast<uint4*>(p.y_f16) + ((tile * p.n + t) * 16 + 4 * ublk) * kTcTile + row;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            uint4 v;
            v.x = emit ? tc::pack_half2(h[8 * q], h[8 * q + 1]) : 0u;
            v.y = emit ? tc::pack_half2(h[8 * q + 2], h[8 * q + 3]) : 0u;
            v.z = emit ? tc::pack_half2(h[8 * q + 4], h[8 * q + 5]) : 0u;
            v.w = emit ? tc::pack_half2(h[8 * q + 6], h[8 * q + 7]) : 0u;
            dst[q * kTcTile] = v;
          }
        }
        emit_prev = emit;
      }
      if (kLast && p.nt > 0) {
        // the tile's last logits; every thread waits for that product because the next tile's prologue overwrites A_h
        if (ublk == 0) {
          read_logits(nf & 1, emit_prev);
          emit_probs(t_end - 1);
        } else {
          mbar_acquire(&bars[kBarF], nf & 1);
        }
        ++nf;
      }
      if (ok) {
        float4* dst = reinterpret_cast<float4*>(p.h_out + s * kHidden + u0);
#pragma unroll
        for (int i = 0; i < kTcUnits / 4; ++i) dst[i] = make_float4(h[4 * i], h[4 * i + 1], h[4 * i + 2], h[4 * i + 3]);
      }
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == kMmaWarp) tc::tmem_dealloc(tmem, 512);
}

static size_t gru_tc_smem_bytes(int kxw, bool last, int nbuf) {
  return static_cast<size_t>(768) * (kxw + kHidden) + static_cast<size_t>(nbuf) * (kxw / 8) * tc::kTileChunkBytes +
         sizeof(float) * 384 + (last ? kFcOperandBytes + sizeof(float) * (4 * 6 + kTcMaxClasses) * kTcTile : 0) +
         kNumBars * sizeof(uint64_t) + 16;
}
static size_t max_dynamic_smem(int device) {
  int v = 0;
  if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, device) != cudaSuccess) return 0;
  return static_cast<size_t>(v);
}
// x buffers the kernel can keep for a layer with `kxw` operand columns: 2, 1, or 0 (the layer does not fit at all)
static int gru_tc_x_buffers(int kxw, bool last, int device) {
  const size_t cap = max_dynamic_smem(device);
  if (gru_tc_smem_bytes(kxw, last, 2) <= cap) return 2;
  if (gru_tc_smem_bytes(kxw, last, 1) <= cap) return 1;
  return 0;
}
// the x product of a first layer of `in_dim` inputs can be split (x_hi/x_lo operand, Wx_hi/Wx_lo weights)
bool gru_tc_can_split(int in_dim, bool last, int device) {
  const int kx = (in_dim + 15) / 16 * 16;
  return gru_tc_x_buffers(2 * kx, last, device) > 0;
}
// first layer: weights + at least one x buffer; the layers above (128 inputs through TMEM) always fit
bool gru_tc_layer_fits(int in_dim, bool split, bool last, int device) {
  const int kx = (in_dim + 15) / 16 * 16;
  return gru_tc_x_buffers(split ? 2 * kx : kx, last, device) > 0;
}

// Pack one layer's TF kernels into the fp16 canonical [384, kxw+128] B operand: [Wx_hi | Wx_lo (split) | Wh].
void pack_tc_weights(const float* gates_kernel, const float* cand_kernel, int in_dim, bool split, std::vector<__half>* out,
                     int* kx_out, int* kxw_out) {
  const int kx = (in_dim + 15) / 16 * 16;
  const int kxw = split ? 2 * kx : kx;
  const int ktot = kxw + kHidden;
  out->assign(static_cast<size_t>(384) * ktot, __float2half_rn(0.0f));
  unsigned char* base = reinterpret_cast<unsigned char*>(out->data());
  for (int n = 0; n < 384; ++n)
    for (int k = 0; k < ktot; ++k) {
      int src_row;
      bool lo = false;
      if (k < kxw) {
        const int kk = k % kx;
        lo = k >= kx;
        if (kk >= in_dim) continue;
        src_row = kk;
      } else {
        src_row = in_dim + (k - kxw);
      }
      const float v = n < 2 * kHidden ? gates_kernel[static_cast<size_t>(src_row) * 2 * kHidden + n]
                                      : cand_kernel[static_cast<size_t>(src_row) * kHidden + (n - 2 * kHidden)];
      const __half hi = __float2half_rn(v);
      const __half val = lo ? __float2half_rn(v - __half2float(hi)) : hi;
      *reinterpret_cast<__half*>(base + tc::canon_offset(n, k, ktot)) = val;
    }
  *kx_out = kx;
  *kxw_out = kxw;
}

// Callers that hold x as row-major fp32 [S, n, in_dim] (kws_gru_forward): the row-tiled fp16 operand the kernel copies,
// [tile][t][x_hi chunks | x_lo chunks (split)][128 streams][8].  The streaming and deployment paths never run this: their
// front end writes the operand itself.
__global__ void __launch_bounds__(256)
tc_pack_x_kernel(const float* __restrict__ x, long S, int n, int in_dim, int nc, int split, uint4* __restrict__ out) {
  const long ntiles = (S + kTcTile - 1) / kTcTile;
  const long total = ntiles * n * nc * kTcTile;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int row = static_cast<int>(i & (kTcTile - 1));
    long r = i >> 7;
    const int c = static_cast<int>(r % nc);
    r /= nc;
    const int t = static_cast<int>(r % n);
    const long tile = r / n;
    const long s = tile * kTcTile + row;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = 8 * c + j;
      v[j] = (s < S && k < in_dim) ? __ldg(x + (s * n + t) * static_cast<long>(in_dim) + k) : 0.0f;
    }
    uint4 hi, lo;
    tc::split_half8(v, &hi, &lo);
    const long base = (tile * n + t) * static_cast<long>(split ? 2 * nc : nc);
    out[(base + c) * kTcTile + row] = hi;
    if (split) out[(base + nc + c) * kTcTile + row] = lo;
  }
}

int launch_gru_tc(kws_model* m, const GruArgs& a, float* hand_off, cudaStream_t st) {
  const int L = m->cfg.num_layers;
  const long ntiles = ceil_div(a.S, kTcTile);
  const size_t per_buf = static_cast<size_t>(ntiles) * kTcTile * a.n * kHidden;     // halves (whole tiles)
  __half* seq = reinterpret_cast<__half*>(hand_off);
  // layer 0's operand: written by the front end (x_tiled), or packed here from the caller's row-major fp32 x
  const unsigned char* x0 = reinterpret_cast<const unsigned char*>(a.x);
  if (!a.x_tiled) {
    const int nc = m->layer[0].tc_kx / 8;
    const bool split = m->layer[0].tc_kxw != m->layer[0].tc_kx;
    const size_t need = static_cast<size_t>(ntiles) * a.n * (m->layer[0].tc_kxw / 8) * tc::kTileChunkBytes;
    const int rc = grow_scratch(&m->tc_xt, &m->tc_xt_bytes, need, "x operand scratch");
    if (rc != KWS_OK) return rc;
    const long total = ntiles * a.n * nc * kTcTile;
    const long blocks = std::min<long>(ceil_div(total, 256), static_cast<long>(sm_count()) * 16);
    tc_pack_x_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(a.x, a.S, a.n, m->layer[0].in_dim, nc, split ? 1 : 0,
                                                                    static_cast<uint4*>(m->tc_xt));
    KWS_LAUNCH_OK("tc_pack_x_kernel");
    x0 = static_cast<const unsigned char*>(m->tc_xt);
  }
  // frames [t0, t0 + nt) of layer l on stream `cs`; `head` = the first chunk of the sequence (incoming state, VAD reset)
  auto launch_layer = [&](int l, int t0, int nt, bool head, cudaStream_t cs) -> int {
    const bool last = l == L - 1;
    GruTcParams p;
    p.kx = m->layer[l].tc_kx;
    p.kxw = m->layer[l].tc_kxw;
    p.nbuf = l == 0 ? gru_tc_x_buffers(p.kxw, last, m->device) : 1;
    if (p.nbuf == 0)
      return fail(KWS_ERR_UNSUPPORTED, "layer %d (%d inputs) does not fit the tensor-core recurrent kernel's shared memory", l,
                  m->layer[l].in_dim);
    p.S = a.S;
    p.n = a.n;
    p.t0 = t0;
    p.nt = nt;
    p.x_tiles = l == 0 ? x0 : nullptr;
    p.x_f16 = l == 0 ? nullptr : seq + ((l - 1) & 1) * per_buf;
    p.y_f16 = last ? nullptr : seq + (l & 1) * per_buf;
    p.wpack = static_cast<const __half*>(m->layer[l].tc_wpack);
    p.bias = m->layer[l].tc_bias;
    p.h_out = a.state_out + static_cast<long>(l) * a.S * kHidden;
    p.h_in = head ? a.state_in + static_cast<long>(l) * a.S * kHidden : p.h_out;
    p.seq_len = a.seq_len;
    p.zero_state = head ? a.zero_state : nullptr;
    p.C = m->cfg.num_classes;
    p.probs = a.probs;
    p.logits = a.logits;
    for (int j = 0; j < kHidden; ++j)
      for (int c = 0; c < kTcMaxClasses; ++c) p.fcw[j * kTcMaxClasses + c] = c < m->cfg.num_classes ? m->fc_w_host[j * m->cfg.num_classes + c] : 0.0f;
    for (int c = 0; c < kTcMaxClasses; ++c) p.fcb[c] = c < m->cfg.num_classes ? m->fc_b_host[c] : 0.0f;
    const size_t smem = gru_tc_smem_bytes(p.kxw, last, l == 0 ? p.nbuf : 0);
    const long blocks = ntiles < sm_count() ? ntiles : sm_count();
    auto launch = [&](auto kernel) -> int {
      KWS_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
      kernel<<<static_cast<unsigned>(blocks), kTcThreads, smem, cs>>>(p);
      return KWS_OK;
    };
    // straight-line issue code for the shapes of the deployment model; another mel count takes its trip counts from p
    const bool mel40 = p.kx == 48 && p.kxw == 96;
    int rc;
    if (l > 0) rc = last ? launch(gru_tc_kernel<true, false, 8>) : launch(gru_tc_kernel<false, false, 8>);
    else if (last) rc = mel40 ? launch(gru_tc_kernel<true, true, 3>) : launch(gru_tc_kernel<true, true, 0>);
    else rc = mel40 ? launch(gru_tc_kernel<false, true, 3>) : launch(gru_tc_kernel<false, true, 0>);
    if (rc != KWS_OK) return rc;
    KWS_LAUNCH_OK("gru_tc_kernel");
    return KWS_OK;
  };

  // Small batches of long sequences (BASELINE config 2: 4096 utterances x 298 frames = 32 tiles on 148 SMs): the two
  // layers are pipelined in time chunks on two streams -- layer 1 runs chunk c while layer 0 runs chunk c + 1 -- so
  // twice as many SMs work.  The recurrence itself is sequential; large batches fill the GPU without this.
  constexpr int kChunk = 64;                                   // multiple of 4: the batched probability stores stay aligned
  const bool pipelined = L == 2 && 2 * ntiles <= sm_count() && a.n >= 2 * kChunk;
  if (!pipelined) {
    for (int l = 0; l < L; ++l) {
      const int rc = launch_layer(l, 0, a.n, true, st);
      if (rc != KWS_OK) return rc;
    }
    return KWS_OK;
  }
  if (!m->aux_stream) KWS_CUDA_OK(cudaStreamCreateWithFlags(&m->aux_stream, cudaStreamNonBlocking));
  const int nchunks = a.n / kChunk;                            // the last chunk takes the remainder
  while (static_cast<int>(m->aux_events.size()) < nchunks + 1) {
    cudaEvent_t e;
    KWS_CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    m->aux_events.push_back(e);
  }
  for (int c = 0; c < nchunks; ++c) {
    const int t0 = c * kChunk;
    const int nt = c == nchunks - 1 ? a.n - t0 : kChunk;
    int rc = launch_layer(0, t0, nt, c == 0, st);
    if (rc != KWS_OK) return rc;
    KWS_CUDA_OK(cudaEventRecord(m->aux_events[c], st));
    KWS_CUDA_OK(cudaStreamWaitEvent(m->aux_stream, m->aux_events[c], 0));
    rc = launch_layer(1, t0, nt, c == 0, m->aux_stream);
    if (rc != KWS_OK) return rc;
  }
  KWS_CUDA_OK(cudaEventRecord(m->aux_events[nchunks], m->aux_stream));
  KWS_CUDA_OK(cudaStreamWaitEvent(st, m->aux_events[nchunks], 0));
  return KWS_OK;
}

}  // namespace kws
