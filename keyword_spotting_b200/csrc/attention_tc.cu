// Dense layers of the attention_ctc forward pass on the 5th-generation tensor cores (models/attention_ctc.py:61-70
// feed_forward, :28-58 the q/k/v projections, :92-98 input_linear_trans).
//
//   Y[r, n] = act( sum_k A[r, k] W[k, n] + bias[n] ) (+ pe[r % Tp, n])          A fp32 [rows, K], Y fp32 [rows, N]
//
// In a variable-length batch a tile whose 128 rows all lie at or past their utterances' T'_b loads and stores nothing.
//
// One CTA = a [128 rows, 128 columns] output tile, three CTAs per SM.  K is walked in chunks of 64: the CTA's 256 threads
// read the A chunk from HBM (coalesced 16-byte loads), split every value into two fp16 terms (x = hi + lo, exact to
// 2^-22) and store both in the tcgen05 K-major canonical layout in shared memory; the weight chunk arrives pre-split and
// pre-packed (hi | lo, packed once at model creation) as one linear 32 KB copy.  One elected thread issues
// A_hi W_hi + A_lo W_hi + A_hi W_lo  (12 tcgen05.mma kind::f16 per chunk, SS form, fp32 accumulation in 128 TMEM
// columns): fp32-grade results (the dropped lo x lo term is 2^-22 relative), which is what the 1e-4 parity of this model's
// tests needs -- a single fp16 rounding of the layer-normed activations would cost 5e-4.  Epilogue: TMEM -> registers,
// bias / relu, through a shared-memory transpose to 64-byte row pieces (+ the positional encoding), fp32 to HBM.
// The chunk loop is not pipelined inside a CTA; the other two CTAs of the SM fill its load and store phases.
#include <vector>

#include "common.cuh"
#include "tc05.cuh"

namespace kws {

constexpr int kAlTile = 128;                     // rows and columns of an output tile
constexpr int kAlKc = 64;                        // K elements per chunk
constexpr int kAlThreads = 256;
constexpr int kAlLboA = 144;                     // A operand: 128 + 16 bytes between K-adjacent core matrices (bank spread of the 8-byte stores)
constexpr int kAlSboA = (kAlKc / 8) * kAlLboA;   // 1152
constexpr int kAlPartA = (kAlTile / 8) * kAlSboA;   // 18432 bytes per fp16 part of the A chunk
constexpr int kAlSboW = (kAlKc / 8) * 128;       // 1024: the weights are packed densely (linear copy)
constexpr int kAlPartW = (kAlTile / 8) * kAlSboW;   // 16384
constexpr int kAlSmem = 2 * kAlPartA + 2 * kAlPartW;

template <bool kRelu, bool kAddPe>
__global__ void __launch_bounds__(kAlThreads, 3)
att_linear_tc_kernel(const float* __restrict__ A, const unsigned char* __restrict__ wpack, const float* __restrict__ bias,
                     const float* __restrict__ pe, int Tp, AttLens lens, long rows, int K, int nchunks, int N,
                     float* __restrict__ Y) {
  if (!lens.tile_live(Tp, rows, blockIdx.x * static_cast<long>(kAlTile), kAlTile)) return;   // padding rows only
  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* sA = smem;                               // [hi | lo] x kAlPartA
  unsigned char* sW = smem + 2 * kAlPartA;                // [hi | lo] x kAlPartW
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long r0 = blockIdx.x * static_cast<long>(kAlTile);
  const int nt = blockIdx.y;

  if (warp == 0) tc::tmem_alloc(&tmem_slot, 128);
  if (tid == 0) {
    tc::mbar_init(&bar, 1);
    tc::mbar_fence_init();
  }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = tmem_slot;
  const uint32_t idesc = tc::idesc_f16(128, 128);
  const uint64_t adesc = tc::smem_desc(tc::smem_u32(sA), kAlLboA, kAlSboA);
  const uint64_t wdesc = tc::smem_desc(tc::smem_u32(sW), 128, kAlSboW);

  // this thread's eight 16-byte pieces of an A chunk: 16 consecutive threads read the 256 contiguous bytes of a row.  The
  // pieces of chunk kc + 1 are requested before the MMAs of chunk kc are issued, so HBM latency runs under them.
  constexpr int kPieces = kAlTile * (kAlKc / 4) / kAlThreads;
  float4 areg[kPieces];
  auto load_a = [&](int kc) {
#pragma unroll
    for (int j = 0; j < kPieces; ++j) {
      const int i = tid + j * kAlThreads;
      const int row = i >> 4, q = i & 15;
      const int k = kc * kAlKc + 4 * q;
      const long gr = r0 + row;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (gr < rows) {
        const float* src = A + gr * K + k;
        if (k + 3 < K) {
          v = __ldg(reinterpret_cast<const float4*>(src));
        } else {
          if (k < K) v.x = __ldg(src);
          if (k + 1 < K) v.y = __ldg(src + 1);
          if (k + 2 < K) v.z = __ldg(src + 2);
        }
      }
      areg[j] = v;
    }
  };
  load_a(0);
  for (int kc = 0; kc < nchunks; ++kc) {
    if (kc > 0) {                                          // the previous chunk's MMAs have read both buffers
      tc::mbar_wait(&bar, (kc - 1) & 1);
      tc::fence_after_sync();
    }
    {
      const uint4* wsrc = reinterpret_cast<const uint4*>(wpack + (static_cast<size_t>(nt) * nchunks + kc) * (2 * kAlPartW));
#pragma unroll
      for (int i = tid; i < 2 * kAlPartW / 16; i += kAlThreads) reinterpret_cast<uint4*>(sW)[i] = __ldg(wsrc + i);
    }
#pragma unroll
    for (int j = 0; j < kPieces; ++j) {
      const int i = tid + j * kAlThreads;
      const int row = i >> 4, q = i & 15;
      const float4 v = areg[j];
      const __half2 h01 = __floats2half2_rn(v.x, v.y), h23 = __floats2half2_rn(v.z, v.w);
      const float2 b01 = __half22float2(h01), b23 = __half22float2(h23);
      const uint32_t off = (row >> 3) * kAlSboA + (q >> 1) * kAlLboA + (row & 7) * 16 + (q & 1) * 8;
      *reinterpret_cast<uint2*>(sA + off) = make_uint2(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23));
      *reinterpret_cast<uint2*>(sA + kAlPartA + off) =
          make_uint2(tc::pack_half2(v.x - b01.x, v.y - b01.y), tc::pack_half2(v.z - b23.x, v.w - b23.y));
    }
    if (kc + 1 < nchunks) load_a(kc + 1);
    tc::fence_proxy_async();                               // generic-proxy stores -> MMA operand fetch
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) {
      tc::fence_after_sync();
      if (tc::elect_one()) {
#pragma unroll
        for (int k16 = 0; k16 < kAlKc / 16; ++k16) {
          const uint64_t a_hi = adesc + ((2 * k16 * kAlLboA) >> 4), a_lo = a_hi + (kAlPartA >> 4);
          const uint64_t w_hi = wdesc + ((2 * k16 * 128) >> 4), w_lo = w_hi + (kAlPartW >> 4);
          tc::mma_ss(tmem, a_hi, w_hi, idesc, kc > 0 || k16 > 0);
          tc::mma_ss(tmem, a_lo, w_hi, idesc, true);
          tc::mma_ss(tmem, a_hi, w_lo, idesc, true);
        }
        tc::commit(&bar);
      }
    }
  }
  tc::mbar_wait(&bar, (nchunks - 1) & 1);
  tc::fence_after_sync();

  // ---- epilogue: warp = (TMEM lane quarter, half of the tile's columns); the A buffers are free and serve as staging
  const int q4 = warp & 3, chalf = warp >> 2;
  const uint32_t lane_sel = static_cast<uint32_t>(32 * q4) << 16;
  float* stage = reinterpret_cast<float*>(sA) + warp * (32 * 20);          // [32 rows][16 cols], row stride 80 bytes
  const long rbase = r0 + 32 * q4;
#pragma unroll 1
  for (int ch = 0; ch < 4; ++ch) {
    const int c0 = 64 * chalf + 16 * ch;                                   // column of the tile
    const int n0 = nt * kAlTile + c0;
    uint32_t v[16];
    tc::ld16(tmem + lane_sel + c0, v);
    tc::wait_ld();
#pragma unroll
    for (int i = 0; i < 16; i += 4) {
      const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias + n0 + i));
      float o0 = __uint_as_float(v[i]) + b4.x, o1 = __uint_as_float(v[i + 1]) + b4.y;
      float o2 = __uint_as_float(v[i + 2]) + b4.z, o3 = __uint_as_float(v[i + 3]) + b4.w;
      if (kRelu) {
        o0 = fmaxf(o0, 0.0f); o1 = fmaxf(o1, 0.0f); o2 = fmaxf(o2, 0.0f); o3 = fmaxf(o3, 0.0f);
      }
      *reinterpret_cast<float4*>(stage + lane * 20 + i) = make_float4(o0, o1, o2, o3);
    }
    __syncwarp();
#pragma unroll
    for (int itr = 0; itr < 4; ++itr) {                                    // 4 lanes cover the 64 contiguous bytes of a row
      const int rr = itr * 8 + (lane >> 2), cc = 4 * (lane & 3);
      float4 o4 = *reinterpret_cast<const float4*>(stage + rr * 20 + cc);
      const long grr = rbase + rr;
      if (grr < rows) {
        if (kAddPe) {
          const float4 p4 = __ldg(reinterpret_cast<const float4*>(pe + static_cast<long>(grr % Tp) * N + n0 + cc));
          o4.x += p4.x; o4.y += p4.y; o4.z += p4.z; o4.w += p4.w;
        }
        *reinterpret_cast<float4*>(Y + grr * N + n0 + cc) = o4;
      }
    }
    __syncwarp();
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem, 128);
}

bool att_linear_tc_supported(int K, int N) { return N % kAlTile == 0 && K % 4 == 0 && K >= 4; }

// W [K, N] row-major fp32 (host) -> per (column tile, K chunk): [hi | lo] fp16 in the canonical K-major layout of the
// B operand ([128 rows = output columns, 64 k]), zero beyond K.  Returns the device buffer.
int att_pack_linear(const float* W, int K, int N, unsigned char** out, int* nchunks_out) {
  const int nchunks = (K + kAlKc - 1) / kAlKc;
  const int ntiles = N / kAlTile;
  std::vector<unsigned char> host(static_cast<size_t>(ntiles) * nchunks * 2 * kAlPartW, 0);
  for (int nt = 0; nt < ntiles; ++nt)
    for (int kc = 0; kc < nchunks; ++kc) {
      unsigned char* base = host.data() + (static_cast<size_t>(nt) * nchunks + kc) * (2 * kAlPartW);
      for (int n = 0; n < kAlTile; ++n)
        for (int kk = 0; kk < kAlKc; ++kk) {
          const int k = kc * kAlKc + kk;
          if (k >= K) continue;
          const float w = W[static_cast<size_t>(k) * N + nt * kAlTile + n];
          const __half hi = __float2half_rn(w);
          const __half lo = __float2half_rn(w - __half2float(hi));
          const size_t off = static_cast<size_t>(n / 8) * kAlSboW + static_cast<size_t>(kk / 8) * 128 + (n % 8) * 16 + (kk % 8) * 2;
          *reinterpret_cast<__half*>(base + off) = hi;
          *reinterpret_cast<__half*>(base + kAlPartW + off) = lo;
        }
    }
  *out = nullptr;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(out), host.size());
  if (e != cudaSuccess) return fail(KWS_ERR_ALLOC, "cudaMalloc(%zu) failed: %s", host.size(), cudaGetErrorString(e));
  KWS_CUDA_OK(cudaMemcpy(*out, host.data(), host.size(), cudaMemcpyHostToDevice));
  *nchunks_out = nchunks;
  return KWS_OK;
}

int launch_att_linear_tc(const float* A, const unsigned char* wpack, int nchunks, const float* bias, const float* pe, int Tp,
                         AttLens lens, long rows, int K, int N, bool relu, bool add_pe, float* Y, cudaStream_t st) {
  if (rows <= 0) return KWS_OK;
  dim3 grid(static_cast<unsigned>(ceil_div(rows, kAlTile)), static_cast<unsigned>(N / kAlTile));
  auto launch = [&](auto kernel) -> int {
    KWS_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kAlSmem));
    kernel<<<grid, kAlThreads, kAlSmem, st>>>(A, wpack, bias, pe, Tp, lens, rows, K, nchunks, N, Y);
    return KWS_OK;
  };
  int rc;
  if (relu) rc = add_pe ? launch(att_linear_tc_kernel<true, true>) : launch(att_linear_tc_kernel<true, false>);
  else rc = add_pe ? launch(att_linear_tc_kernel<false, true>) : launch(att_linear_tc_kernel<false, false>);
  if (rc != KWS_OK) return rc;
  KWS_LAUNCH_OK("att_linear_tc_kernel");
  return KWS_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Multi-head attention core on the tensor cores (models/attention_ctc.py:28-58): per (utterance, head)
//     O = softmax(Q K^T / sqrt(16)) V        over ALL T'_b keys of the utterance (no mask), T'_b <= 400, head size 16.
// Rows are laid out with stride T' (the batch's longest); utterance b has its own T'_b <= T' rows and keys, and CTAs of
// utterances with T'_b > 400 return at once (the FFMA core takes those).
// One CTA per (utterance, head); K and V^T are split into fp16 hi/lo once and stay in shared memory as B operands, the
// CTA then walks the utterance's query tiles of 128 rows:
//   S = Q K^T   6 tcgen05.mma (3 hi/lo products x N = 256 + the rest, K = 16) into T' columns of TMEM;
//   pass 1      every thread reads its row's scores (two warps per TMEM lane quarter, half of the keys each): row maximum;
//   pass 2      re-read, p = 2^(s - max), row sum; p is written back IN PLACE as the next product's A operand: the 16 score
//               columns of a key group become 8 columns of fp16(p) and 8 columns of its rounding remainder;
//   O = P V     75 tcgen05.mma (3 products x 25 key groups, N = 16, TS form) into 16 more TMEM columns;
//   O / sum -> HBM (64 bytes per query row).
// fp32-grade throughout (the dropped lo x lo terms are 2^-22 relative): the model's 1e-4 parity tests are unchanged.
constexpr int kAcThreads = 256;
constexpr int kAcD = 16;
constexpr int kAcMaxKeys = kAttCoreTcMaxKeys;    // T' padded to a multiple of 16; TMEM: 400 score columns + 16 for O
constexpr int kAcSboK = 2 * 128;                 // K operand [keys, 16]: two K-adjacent core matrices per 8-key group
constexpr int kAcPartK = (kAcMaxKeys / 8) * kAcSboK;      // 12800
constexpr int kAcSboV = (kAcMaxKeys / 8) * 128;  // V^T operand [16, keys]: 6400 between the two 8-row groups
constexpr int kAcPartV = 2 * kAcSboV;            // 12800
constexpr int kAcPartQ = (128 / 8) * kAcSboK;    // 4096
constexpr int kAcColO = kAcMaxKeys;

__device__ __forceinline__ float ex2_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__global__ void __launch_bounds__(kAcThreads, 1)
att_core_tc_kernel(const float* __restrict__ qkv, int Tp, int heads, AttLens lens, float* __restrict__ out) {
  const long b = blockIdx.x / heads;
  const int Tb = lens.rows_of(b);                               // this utterance's keys and queries; Tp is the row stride
  if (Tb > kAcMaxKeys) return;
  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* sK = smem;                                      // [hi | lo] x kAcPartK
  unsigned char* sV = sK + 2 * kAcPartK;
  unsigned char* sQ = sV + 2 * kAcPartV;
  __shared__ float sMax[2][128], sSum[2][128];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = heads * kAcD;
  const int h = blockIdx.x % heads;
  const float* base = qkv + b * Tp * 3L * N + h * kAcD;
  const int Kp = (Tb + 15) & ~15;                               // keys padded to whole MMA K steps
  const int groups = Kp / 16;
  const float scale = rsqrtf(static_cast<float>(kAcD)) * 1.4426950408889634f;     // 1/sqrt(d), in log2 units

  if (warp == 0) tc::tmem_alloc(&tmem_slot, 512);
  if (tid == 0) {
    tc::mbar_init(&bar, 1);
    tc::mbar_fence_init();
  }
  // ---- K and V^T of this head, split into hi / lo fp16 (zero rows past T')
  for (int j = tid; j < Kp; j += kAcThreads) {
    float kf[16], vf[16];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float4 k4 = make_float4(0.f, 0.f, 0.f, 0.f), v4 = k4;
      if (j < Tb) {
        k4 = __ldg(reinterpret_cast<const float4*>(base + static_cast<long>(j) * 3 * N + N) + c);
        v4 = __ldg(reinterpret_cast<const float4*>(base + static_cast<long>(j) * 3 * N + 2 * N) + c);
      }
      kf[4 * c] = k4.x; kf[4 * c + 1] = k4.y; kf[4 * c + 2] = k4.z; kf[4 * c + 3] = k4.w;
      vf[4 * c] = v4.x; vf[4 * c + 1] = v4.y; vf[4 * c + 2] = v4.z; vf[4 * c + 3] = v4.w;
    }
#pragma unroll
    for (int c = 0; c < 2; ++c) {                                // K: 8 consecutive d of key j are one 16-byte row piece
      const float v8[8] = {kf[8 * c], kf[8 * c + 1], kf[8 * c + 2], kf[8 * c + 3], kf[8 * c + 4], kf[8 * c + 5], kf[8 * c + 6], kf[8 * c + 7]};
      uint4 hi, lo;
      tc::split_half8(v8, &hi, &lo);
      const uint32_t off = (j >> 3) * kAcSboK + c * 128 + (j & 7) * 16;
      *reinterpret_cast<uint4*>(sK + off) = hi;
      *reinterpret_cast<uint4*>(sK + kAcPartK + off) = lo;
    }
#pragma unroll
    for (int d = 0; d < 16; ++d) {                               // V^T: element (d, key j)
      const __half hi = __float2half_rn(vf[d]);
      const __half lo = __float2half_rn(vf[d] - __half2float(hi));
      const uint32_t off = (d >> 3) * kAcSboV + (j >> 3) * 128 + (d & 7) * 16 + (j & 7) * 2;
      *reinterpret_cast<__half*>(sV + off) = hi;
      *reinterpret_cast<__half*>(sV + kAcPartV + off) = lo;
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = tmem_slot;
  const uint64_t kdesc = tc::smem_desc(tc::smem_u32(sK), 128, kAcSboK);
  const uint64_t vdesc = tc::smem_desc(tc::smem_u32(sV), 128, kAcSboV);
  const uint64_t qdesc = tc::smem_desc(tc::smem_u32(sQ), 128, kAcSboK);
  const int n1 = Kp < 256 ? Kp : 256, n2 = Kp - n1;              // the score product as one or two MMAs along N
  const uint32_t idesc1 = tc::idesc_f16(128, n1), idesc2 = tc::idesc_f16(128, n2 > 0 ? n2 : 16), idesc_o = tc::idesc_f16(128, 16);

  const int q4 = warp & 3, ch = warp >> 2;                       // TMEM lane quarter; which half of the key groups
  const int row = 32 * q4 + lane;
  const uint32_t lane_sel = static_cast<uint32_t>(32 * q4) << 16;
  const int g_split = (groups + 1) / 2;
  const int g_begin = ch == 0 ? 0 : g_split, g_end = ch == 0 ? g_split : groups;
  uint32_t phase = 0;

  for (int i0 = 0; i0 < Tb; i0 += 128) {
    // ---- Q tile: row = query i0 + r, scaled to log2 units, hi / lo
    if (tid < 128) {
      const int i = i0 + tid;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        float v8[8];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          float4 q4v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (i < Tb) q4v = __ldg(reinterpret_cast<const float4*>(base + static_cast<long>(i) * 3 * N) + 2 * c + e);
          v8[4 * e] = q4v.x * scale; v8[4 * e + 1] = q4v.y * scale; v8[4 * e + 2] = q4v.z * scale; v8[4 * e + 3] = q4v.w * scale;
        }
        uint4 hi, lo;
        tc::split_half8(v8, &hi, &lo);
        const uint32_t off = (tid >> 3) * kAcSboK + c * 128 + (tid & 7) * 16;
        *reinterpret_cast<uint4*>(sQ + off) = hi;
        *reinterpret_cast<uint4*>(sQ + kAcPartQ + off) = lo;
      }
    }
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    // ---- S = Q K^T (K = 16: one step): Qh Kh + Ql Kh + Qh Kl
    if (warp == 0) {
      tc::fence_after_sync();
      if (tc::elect_one()) {
        const uint64_t ql = qdesc + (kAcPartQ >> 4), kl = kdesc + (kAcPartK >> 4);
        tc::mma_ss(tmem, qdesc, kdesc, idesc1, false);
        tc::mma_ss(tmem, ql, kdesc, idesc1, true);
        tc::mma_ss(tmem, qdesc, kl, idesc1, true);
        if (n2 > 0) {
          const uint64_t koff = static_cast<uint64_t>((256 / 8) * kAcSboK) >> 4;      // key rows 256..
          tc::mma_ss(tmem + 256, qdesc, kdesc + koff, idesc2, false);
          tc::mma_ss(tmem + 256, ql, kdesc + koff, idesc2, true);
          tc::mma_ss(tmem + 256, qdesc, kl + koff, idesc2, true);
        }
        tc::commit(&bar);
      }
    }
    tc::mbar_wait(&bar, phase & 1);
    ++phase;
    tc::fence_after_sync();
    // (a warp whose 32 query rows all lie past T' -- three of the four lane quarters of the last tile -- skips both passes:
    // its rows of P stay garbage, which only reaches its own, never stored, rows of O)
    const bool warp_live = i0 + 32 * q4 < Tb;
    const int g_tail = (Tb & 15) ? groups - 1 : groups;          // the one key group with padded keys, if any
    // ---- pass 1: row maximum over this warp's key groups
    float mx = -INFINITY;
    if (warp_live) {
      for (int g = g_begin; g < g_end; ++g) {
        uint32_t v[16];
        tc::ld16(tmem + lane_sel + 16 * g, v);
        tc::wait_ld();
        if (g < g_tail) {
#pragma unroll
          for (int e = 0; e < 16; ++e) mx = fmaxf(mx, __uint_as_float(v[e]));
        } else {
#pragma unroll
          for (int e = 0; e < 16; ++e)
            if (16 * g + e < Tb) mx = fmaxf(mx, __uint_as_float(v[e]));
        }
      }
    }
    sMax[ch][row] = mx;
    __syncthreads();
    mx = fmaxf(sMax[0][row], sMax[1][row]);
    // ---- pass 2: p = 2^(s - max) back into the same columns as the A operand of the next product (hi | lo per key group)
    float sum = 0.0f;
    if (warp_live) {
      for (int g = g_begin; g < g_end; ++g) {
        uint32_t v[16];
        tc::ld16(tmem + lane_sel + 16 * g, v);
        tc::wait_ld();
        uint32_t ph[8], pl[8];
#pragma unroll
        for (int e = 0; e < 16; e += 2) {
          float p0 = ex2_fast(__uint_as_float(v[e]) - mx), p1 = ex2_fast(__uint_as_float(v[e + 1]) - mx);
          if (g >= g_tail) {                                     // padded keys carry no weight
            if (16 * g + e >= Tb) p0 = 0.0f;
            if (16 * g + e + 1 >= Tb) p1 = 0.0f;
          }
          sum += p0 + p1;
          const __half2 hh = __floats2half2_rn(p0, p1);
          const float2 bb = __half22float2(hh);
          ph[e / 2] = *reinterpret_cast<const uint32_t*>(&hh);
          pl[e / 2] = tc::pack_half2(p0 - bb.x, p1 - bb.y);
        }
        tc::st8(tmem + lane_sel + 16 * g, ph);
        tc::st8(tmem + lane_sel + 16 * g + 8, pl);
      }
    }
    sSum[ch][row] = sum;
    tc::wait_st();
    tc::fence_before_sync();
    __syncthreads();
    // ---- O = P V: per key group  Ph Vh + Pl Vh + Ph Vl
    if (warp == 0) {
      tc::fence_after_sync();
      if (tc::elect_one()) {
        const uint64_t vl = vdesc + (kAcPartV >> 4);
        for (int g = 0; g < groups; ++g) {
          const uint64_t step = static_cast<uint64_t>(g) * ((2 * 128) >> 4);
          tc::mma_ts(tmem + kAcColO, tmem + 16 * g, vdesc + step, idesc_o, g > 0);
          tc::mma_ts(tmem + kAcColO, tmem + 16 * g + 8, vdesc + step, idesc_o, true);
          tc::mma_ts(tmem + kAcColO, tmem + 16 * g, vl + step, idesc_o, true);
        }
        tc::commit(&bar);
      }
    }
    tc::mbar_wait(&bar, phase & 1);
    ++phase;
    tc::fence_after_sync();
    if (ch == 0) {
      uint32_t v[16];
      tc::ld16(tmem + lane_sel + kAcColO, v);
      tc::wait_ld();
      const int i = i0 + row;
      if (i < Tb) {
        const float inv = 1.0f / (sSum[0][row] + sSum[1][row]);
        float4* dst = reinterpret_cast<float4*>(out + (b * Tp + i) * N + h * kAcD);
#pragma unroll
        for (int c = 0; c < 4; ++c)
          dst[c] = make_float4(__uint_as_float(v[4 * c]) * inv, __uint_as_float(v[4 * c + 1]) * inv,
                               __uint_as_float(v[4 * c + 2]) * inv, __uint_as_float(v[4 * c + 3]) * inv);
      }
    }
    tc::fence_before_sync();
    __syncthreads();                              // the tile's TMEM columns and sQ are reused by the next tile
    tc::fence_after_sync();
  }
  if (warp == 0) tc::tmem_dealloc(tmem, 512);
}

bool att_core_tc_supported(int Tp, int heads, int hidden) { return Tp >= 1 && Tp <= kAcMaxKeys && hidden == heads * kAcD; }

int launch_att_core_tc(const float* qkv, long B, int Tp, int heads, AttLens lens, float* out, cudaStream_t st) {
  if (B <= 0) return KWS_OK;
  constexpr int smem = 2 * kAcPartK + 2 * kAcPartV + 2 * kAcPartQ;
  KWS_CUDA_OK(cudaFuncSetAttribute(att_core_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  att_core_tc_kernel<<<static_cast<unsigned>(B * heads), kAcThreads, smem, st>>>(qkv, Tp, heads, lens, out);
  KWS_LAUNCH_OK("att_core_tc_kernel");
  return KWS_OK;
}

}  // namespace kws
