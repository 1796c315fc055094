// K5 -- OctbitMatMul on the GPU, bit-exact with the reference CPU kernel.
// Reference: OctbitMatMulOp::Compute, octbit/octbit_mat_mul_op.cc:49-183.
//
//   (1) tensor-wide min/max of x                                   (:90-99)
//   (2) u8 quantisation: signed  -> round(x/bscale)+127, bscale = max(-min,max)/127
//                        unsigned-> round(x/bscale),     bscale = max/254   (:101-124)
//   (3) per (row,out): four int32 lanes accumulate sat16(q0*w0+q1*w1)       (:137-170)
//       (_mm_maddubs_epi16 saturates every adjacent-pair sum to int16)
//   (4) out = fp32 sum of the lanes in lane order, -bias if signed, *scale  (:172-179)
//
// Two GEMM back ends behind one entry point:
//   * exact  : CUDA-core dp2a kernel that forms and saturates every pair and keeps the
//              four lanes apart -- any K, the validator for the fast path.
//   * imma   : int8 tensor-core kernel (mma.sync m16n8k32 u8*s8 -> s32) that sums the
//              UNsaturated pairs exactly, plus a sparse correction  sum(sat16(p) - p)
//              over the only pairs that can saturate: same-sign neighbours with
//              |w0|+|w1| >= 129 (q <= 255).  Used for K <= 512, where every partial
//              fp32 lane sum is an integer below 2^24 and therefore the reference's
//              lane-ordered fp32 accumulation equals the exact integer total.
// fp32 steps use __f*_rn intrinsics so nothing is contracted into an FMA (the
// reference is built without -mfma: octbit/op_compile.py:64-72).
#include <cfloat>

#include "common.cuh"
#include "octbit_common.cuh"

namespace kws {

__global__ void octbit_init_kernel(OctbitHeader* h) {
  h->enc_min = enc_float(FLT_MAX);      // std::numeric_limits<float>::max()    (:92)
  h->enc_max = enc_float(-FLT_MAX);     // std::numeric_limits<float>::lowest() (:93)
}

__global__ void __launch_bounds__(256)
octbit_minmax_kernel(const float* __restrict__ x, long n, OctbitHeader* h) {
  float mn = FLT_MAX, mx = -FLT_MAX;
  const long stride = static_cast<long>(gridDim.x) * blockDim.x;
  const long tid = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  const long n4 = n >> 2;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  for (long i = tid; i < n4; i += stride) {
    const float4 v = __ldg(x4 + i);
    if (v.x < mn) mn = v.x;  if (v.x > mx) mx = v.x;     // NaN compares false, as in :96-97
    if (v.y < mn) mn = v.y;  if (v.y > mx) mx = v.y;
    if (v.z < mn) mn = v.z;  if (v.z > mx) mx = v.z;
    if (v.w < mn) mn = v.w;  if (v.w > mx) mx = v.w;
  }
  for (long i = (n4 << 2) + tid; i < n; i += stride) {
    const float v = x[i];
    if (v < mn) mn = v;
    if (v > mx) mx = v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  __shared__ float smn[8], smx[8];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { smn[w] = mn; smx[w] = mx; }
  __syncthreads();
  if (w == 0) {
    mn = l < 8 ? smn[l] : FLT_MAX;
    mx = l < 8 ? smx[l] : -FLT_MAX;
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
      mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (l == 0) {
      atomicMin(&h->enc_min, enc_float(mn));
      atomicMax(&h->enc_max, enc_float(mx));
    }
  }
}

// x[n] fp32 -> q[n] u8 (n % 4 == 0 because K % 64 == 0)
__global__ void __launch_bounds__(256)
octbit_quantize_kernel(const float* __restrict__ x, long n, const OctbitHeader* __restrict__ h,
                       unsigned* __restrict__ q4) {
  const QuantParams p = quant_params(h);
  const long stride = static_cast<long>(gridDim.x) * blockDim.x;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < (n >> 2); i += stride) {
    const float4 v = __ldg(x4 + i);
    q4[i] = quant_one(v.x, p) | (quant_one(v.y, p) << 8) | (quant_one(v.z, p) << 16) |
            (quant_one(v.w, p) << 24);
  }
}

// ---------------------------------------------------------------- exact back end
// One thread per (row, out); 16-byte blocks of q and w -> eight saturated pairs.
__global__ void __launch_bounds__(256)
octbit_gemm_exact_kernel(const unsigned char* __restrict__ q, const signed char* __restrict__ w,
                         const float* __restrict__ bias, float scale_attr, long A, int B, int K,
                         const OctbitHeader* __restrict__ h, float* __restrict__ out) {
  const int o = blockIdx.x * 32 + (threadIdx.x & 31);
  const long a = blockIdx.y * 8L + (threadIdx.x >> 5);
  if (o >= B || a >= A) return;
  const QuantParams p = quant_params(h);
  const uint4* qr = reinterpret_cast<const uint4*>(q + a * K);
  const uint4* wr = reinterpret_cast<const uint4*>(w + static_cast<long>(o) * K);
  int lane[4] = {0, 0, 0, 0};
  for (int blk = 0; blk < K / 16; ++blk) {
    const uint4 qv = qr[blk];
    const uint4 wv = __ldg(wr + blk);
    const unsigned qq[4] = {qv.x, qv.y, qv.z, qv.w};
    const unsigned ww[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int qlo = static_cast<int>(__byte_perm(qq[j], 0u, 0x4140));   // [b0,0,b1,0]
      const int qhi = static_cast<int>(__byte_perm(qq[j], 0u, 0x4342));   // [b2,0,b3,0]
      const int p0 = __dp2a_lo(qlo, static_cast<int>(ww[j]), 0);          // q0*w0 + q1*w1
      const int p1 = __dp2a_hi(qhi, static_cast<int>(ww[j]), 0);          // q2*w2 + q3*w3
      lane[(2 * j) & 3] += sat16(p0);          // pair 2j   -> lane (2j)%4
      lane[(2 * j + 1) & 3] += sat16(p1);      // pair 2j+1 -> lane (2j+1)%4
    }
  }
  const float scale = __fmul_rn(scale_attr, p.bscale);                    // (:108,:117)
  out[a * B + o] = octbit_epilogue(lane[0], lane[1], lane[2], lane[3], p.is_signed, bias[o], scale);
}

// ---------------------------------------------------------------- tensor-core back end
__global__ void __launch_bounds__(256)
octbit_find_candidates_kernel(const signed char* __restrict__ w, int B, int K,
                              int* __restrict__ cand_count, unsigned short* __restrict__ cand) {
  const int half = K / 2;
  const long total = static_cast<long>(B) * half;
  for (long idx = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long>(gridDim.x) * blockDim.x) {
    const int n = static_cast<int>(idx / half);
    const int kp = static_cast<int>(idx - static_cast<long>(n) * half);
    const int w0 = w[static_cast<long>(n) * K + 2 * kp];
    const int w1 = w[static_cast<long>(n) * K + 2 * kp + 1];
    const bool same_sign = (w0 > 0 && w1 > 0) || (w0 < 0 && w1 < 0);
    if (same_sign && abs(w0) + abs(w1) >= 129) {
      const int slot = atomicAdd(cand_count + n, 1);
      cand[static_cast<long>(n) * half + slot] = static_cast<unsigned short>(kp);
    }
  }
}

__device__ __forceinline__ int sat_correction(const unsigned char* __restrict__ qrow,
                                              const signed char* __restrict__ wrow,
                                              const unsigned short* __restrict__ cand, int count) {
  int delta = 0;
  for (int c = 0; c < count; ++c) {
    const int kp = cand[c];
    const int p = static_cast<int>(qrow[2 * kp]) * wrow[2 * kp] +
                  static_cast<int>(qrow[2 * kp + 1]) * wrow[2 * kp + 1];
    delta += sat16(p) - p;
  }
  return delta;
}

// CTA = 4 warps; warp tile 16 rows x 64 cols; CTA tile 64 rows x 64 cols.
__global__ void __launch_bounds__(128)
octbit_gemm_imma_kernel(const unsigned char* __restrict__ q, const signed char* __restrict__ w,
                        const float* __restrict__ bias, float scale_attr, long A, int B, int K,
                        const OctbitHeader* __restrict__ h, const int* __restrict__ cand_count,
                        const unsigned short* __restrict__ cand, float* __restrict__ out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const long m0 = blockIdx.y * 64L + warp * 16;
  const int n0 = blockIdx.x * 64;
  if (m0 >= A) return;
  const long r0 = m0 + g, r1 = m0 + g + 8;
  const bool v0 = r0 < A, v1 = r1 < A;
  const unsigned char* q0 = q + (v0 ? r0 : 0) * K;
  const unsigned char* q1 = q + (v1 ? r1 : 0) * K;
  int acc[8][4];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0;
  const signed char* wn[8];
  bool wv[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int n = n0 + 8 * j + g;
    wv[j] = n < B;
    wn[j] = w + static_cast<long>(wv[j] ? n : 0) * K;
  }
  for (int k0 = 0; k0 < K; k0 += 32) {
    unsigned a[4];
    a[0] = v0 ? *reinterpret_cast<const unsigned*>(q0 + k0 + 4 * t) : 0u;
    a[1] = v1 ? *reinterpret_cast<const unsigned*>(q1 + k0 + 4 * t) : 0u;
    a[2] = v0 ? *reinterpret_cast<const unsigned*>(q0 + k0 + 16 + 4 * t) : 0u;
    a[3] = v1 ? *reinterpret_cast<const unsigned*>(q1 + k0 + 16 + 4 * t) : 0u;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const unsigned b0 = wv[j] ? __ldg(reinterpret_cast<const unsigned*>(wn[j] + k0 + 4 * t)) : 0u;
      const unsigned b1 = wv[j] ? __ldg(reinterpret_cast<const unsigned*>(wn[j] + k0 + 16 + 4 * t)) : 0u;
      mma_u8s8(acc[j], a, b0, b1);
    }
  }
  const QuantParams p = quant_params(h);
  const float scale = __fmul_rn(scale_attr, p.bscale);
  const int half = K / 2;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int n = n0 + 8 * j + 2 * t + (e & 1);
      const long r = (e & 2) ? r1 : r0;
      if (n < B && r < A) {
        const int cnt = cand_count[n];
        int total = acc[j][e];
        if (cnt) total += sat_correction(q + r * K, w + static_cast<long>(n) * K,
                                         cand + static_cast<long>(n) * half, cnt);
        // K <= 512: every fp32 partial sum of the four lanes is an exact integer < 2^24,
        // so the lane-ordered fp32 accumulation of the reference equals float(total).
        out[r * B + n] = octbit_epilogue(total, 0, 0, 0, p.is_signed, bias[n], scale);
      }
    }
  }
}

// ---------------------------------------------------------------- octize (offline recipe)
// octize_weight_int8_signed, octbit/octbit_graph.py:191-215.
__global__ void __launch_bounds__(256)
absmax_kernel(const float* __restrict__ x, long n, unsigned* __restrict__ out_bits) {
  float m = 0.0f;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long>(gridDim.x) * blockDim.x)
    m = fmaxf(m, fabsf(x[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out_bits, __float_as_uint(m));   // non-negative floats order as uints
}

__global__ void __launch_bounds__(128)
octize_kernel(const float* __restrict__ weight, int in_dim, int out_dim, float scale_f,
              signed char* __restrict__ wq_t, float* __restrict__ bias) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= out_dim) return;
  long sum = 0;
  for (int i = 0; i < in_dim; ++i) {
    const float v = rintf(__fdiv_rn(weight[static_cast<long>(i) * out_dim + j], scale_f));  // np.round: half-even
    const int qv = static_cast<int>(v);
    sum += qv;
    wq_t[static_cast<long>(j) * in_dim + i] = static_cast<signed char>(qv);
  }
  bias[j] = static_cast<float>(127.0 * static_cast<double>(sum));
}

static inline size_t align256(size_t v) { return (v + 255) / 256 * 256; }

}  // namespace kws

extern "C" size_t kws_octbit_workspace_bytes(int64_t A, int64_t K) {
  if (A < 0 || K < 0) return 0;
  // header | q[A,K] u8 | cand_count[4096] | cand[4096 * K/2] u16   (B <= 4096 on the fast path)
  return sizeof(kws::OctbitHeader) + kws::align256(static_cast<size_t>(A) * K) +
         kws::align256(4096 * sizeof(int)) + kws::align256(static_cast<size_t>(4096) * (K / 2) * 2);
}

extern "C" int kws_octbit_matmul(const float* x, const int8_t* w, const float* bias, float scale,
                                 int transpose_a, int transpose_b, int64_t A, int64_t B, int64_t K,
                                 float* out, void* workspace, size_t workspace_bytes, void* stream) {
  using namespace kws;
  clear_error();
  // constructor checks, octbit_mat_mul_op.cc:41-46
  KWS_REQUIRE(transpose_b, "b need to be transposed");
  KWS_REQUIRE(!transpose_a, "a cannot to be transposed");
  KWS_REQUIRE(scale > 0, "scale has to be positive");
  // Compute checks, :56-73
  KWS_REQUIRE(A >= 0 && B >= 0 && K >= 0, "negative dimension");
  KWS_REQUIRE(reinterpret_cast<uintptr_t>(w) % 32 == 0, "weight pointer is not 32-byte aligned");
  KWS_REQUIRE(K % 64 == 0, "we need to be 16 aligned. K=%lld", static_cast<long long>(K));
  KWS_REQUIRE(K <= 65536 * 2, "K too large");
  if (A == 0 || B == 0) return KWS_OK;
  KWS_REQUIRE(x && w && bias && out, "NULL tensor pointer");
  KWS_REQUIRE(reinterpret_cast<uintptr_t>(x) % 16 == 0, "x must be 16-byte aligned");
  if (K == 0) {
    // empty contraction: min/max stay at their initial values; the reference then yields
    // (0 - 0) * scale * FLT_MAX/254-ish garbage.  Reject rather than imitate.
    return fail(KWS_ERR_INVALID_ARGUMENT, "K == 0");
  }
  KWS_REQUIRE(workspace != nullptr && workspace_bytes >= kws_octbit_workspace_bytes(A, K),
              "workspace too small: need %zu bytes", kws_octbit_workspace_bytes(A, K));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  OctbitHeader* hdr = reinterpret_cast<OctbitHeader*>(ws);
  unsigned char* q = reinterpret_cast<unsigned char*>(ws + sizeof(OctbitHeader));
  char* after_q = ws + sizeof(OctbitHeader) + align256(static_cast<size_t>(A) * K);
  int* cand_count = reinterpret_cast<int*>(after_q);
  unsigned short* cand = reinterpret_cast<unsigned short*>(after_q + align256(4096 * sizeof(int)));

  const long n = static_cast<long>(A) * K;
  const int sms = sm_count();
  octbit_init_kernel<<<1, 1, 0, st>>>(hdr);
  KWS_LAUNCH_OK("octbit_init_kernel");
  long blocks = ceil_div(n / 4 + 1, 256);
  if (blocks > sms * 8L) blocks = sms * 8L;
  octbit_minmax_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(x, n, hdr);
  KWS_LAUNCH_OK("octbit_minmax_kernel");
  const bool fast = K <= 512 && B <= 4096;
  const bool tc = octbit_tc_supported(A, B, K);       // tcgen05 kind::i8 with the quantiser fused in (octbit_tc.cu)
  if (!tc) {
    octbit_quantize_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(x, n, hdr, reinterpret_cast<unsigned*>(q));
    KWS_LAUNCH_OK("octbit_quantize_kernel");
  }
  if (fast) {
    KWS_CUDA_OK(cudaMemsetAsync(cand_count, 0, sizeof(int) * static_cast<size_t>(B), st));
    long cblocks = ceil_div(B * (K / 2), 256);
    if (cblocks > sms * 8L) cblocks = sms * 8L;
    octbit_find_candidates_kernel<<<static_cast<unsigned>(cblocks), 256, 0, st>>>(
        w, static_cast<int>(B), static_cast<int>(K), cand_count, cand);
    KWS_LAUNCH_OK("octbit_find_candidates_kernel");
    if (tc) return launch_octbit_tc(x, w, bias, scale, A, B, K, hdr, cand_count, cand, out, st);
    dim3 grid(static_cast<unsigned>(ceil_div(B, 64)), static_cast<unsigned>(ceil_div(A, 64)));
    KWS_REQUIRE(ceil_div(A, 64) <= 65535 * 32768LL, "A too large");
    if (grid.y > 65535) {
      // split rows into slabs that respect gridDim.y
      const long slab = 65535L * 64;
      for (long a0 = 0; a0 < A; a0 += slab) {
        const long rows = (A - a0 < slab) ? (A - a0) : slab;
        dim3 g2(grid.x, static_cast<unsigned>(ceil_div(rows, 64)));
        octbit_gemm_imma_kernel<<<g2, 128, 0, st>>>(q + a0 * K, w, bias, scale, rows, static_cast<int>(B),
                                                   static_cast<int>(K), hdr, cand_count, cand, out + a0 * B);
        KWS_LAUNCH_OK("octbit_gemm_imma_kernel");
      }
    } else {
      octbit_gemm_imma_kernel<<<grid, 128, 0, st>>>(q, w, bias, scale, A, static_cast<int>(B),
                                                   static_cast<int>(K), hdr, cand_count, cand, out);
      KWS_LAUNCH_OK("octbit_gemm_imma_kernel");
    }
  } else {
    const long slab = 65535L * 8;
    for (long a0 = 0; a0 < A; a0 += slab) {
      const long rows = (A - a0 < slab) ? (A - a0) : slab;
      dim3 grid(static_cast<unsigned>(ceil_div(B, 32)), static_cast<unsigned>(ceil_div(rows, 8)));
      octbit_gemm_exact_kernel<<<grid, 256, 0, st>>>(q + a0 * K, w, bias, scale, rows, static_cast<int>(B),
                                                    static_cast<int>(K), hdr, out + a0 * B);
      KWS_LAUNCH_OK("octbit_gemm_exact_kernel");
    }
  }
  return KWS_OK;
}

// Forces the exact CUDA-core back end (used by tests to validate the tensor-core path).
extern "C" int kws_octbit_matmul_exact(const float* x, const int8_t* w, const float* bias, float scale,
                                       int64_t A, int64_t B, int64_t K, float* out, void* workspace,
                                       size_t workspace_bytes, void* stream) {
  using namespace kws;
  clear_error();
  KWS_REQUIRE(scale > 0, "scale has to be positive");
  KWS_REQUIRE(K % 64 == 0 && K > 0, "we need to be 16 aligned.");
  KWS_REQUIRE(reinterpret_cast<uintptr_t>(w) % 32 == 0, "weight pointer is not 32-byte aligned");
  if (A == 0 || B == 0) return KWS_OK;
  KWS_REQUIRE(workspace != nullptr && workspace_bytes >= kws_octbit_workspace_bytes(A, K), "workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  OctbitHeader* hdr = reinterpret_cast<OctbitHeader*>(ws);
  unsigned char* q = reinterpret_cast<unsigned char*>(ws + sizeof(OctbitHeader));
  const long n = static_cast<long>(A) * K;
  const int sms = sm_count();
  octbit_init_kernel<<<1, 1, 0, st>>>(hdr);
  long blocks = ceil_div(n / 4 + 1, 256);
  if (blocks > sms * 8L) blocks = sms * 8L;
  octbit_minmax_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(x, n, hdr);
  octbit_quantize_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(x, n, hdr, reinterpret_cast<unsigned*>(q));
  const long slab = 65535L * 8;
  for (long a0 = 0; a0 < A; a0 += slab) {
    const long rows = (A - a0 < slab) ? (A - a0) : slab;
    dim3 grid(static_cast<unsigned>(ceil_div(B, 32)), static_cast<unsigned>(ceil_div(rows, 8)));
    octbit_gemm_exact_kernel<<<grid, 256, 0, st>>>(q + a0 * K, w, bias, scale, rows, static_cast<int>(B),
                                                  static_cast<int>(K), hdr, out + a0 * B);
  }
  KWS_LAUNCH_OK("octbit exact path");
  return KWS_OK;
}

extern "C" int kws_octize_weight(const float* weight, int64_t in_dim, int64_t out_dim, int8_t* wq_t,
                                 float* bias, double* scale_host, void* stream) {
  using namespace kws;
  clear_error();
  KWS_REQUIRE(weight && wq_t && bias && scale_host, "NULL pointer");
  KWS_REQUIRE(in_dim > 0 && out_dim > 0, "empty weight");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // bias[0] doubles as the 4-byte reduction cell before octize_kernel overwrites it
  unsigned* cell = reinterpret_cast<unsigned*>(bias);
  KWS_CUDA_OK(cudaMemsetAsync(cell, 0, sizeof(unsigned), st));
  const long n = static_cast<long>(in_dim) * out_dim;
  long blocks = ceil_div(n, 256);
  if (blocks > sm_count() * 8L) blocks = sm_count() * 8L;
  absmax_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(weight, n, cell);
  KWS_LAUNCH_OK("absmax_kernel");
  float nmax = 0.0f;
  KWS_CUDA_OK(cudaMemcpyAsync(&nmax, cell, sizeof(float), cudaMemcpyDeviceToHost, st));
  KWS_CUDA_OK(cudaStreamSynchronize(st));
  KWS_REQUIRE(nmax > 0.0f, "weight is all zero: scale would be 0");
  const double scale_d = static_cast<double>(nmax) / 127.0;      // nmax / 127.  (:197-198)
  *scale_host = scale_d;
  octize_kernel<<<static_cast<unsigned>(ceil_div(out_dim, 128)), 128, 0, st>>>(
      weight, static_cast<int>(in_dim), static_cast<int>(out_dim), static_cast<float>(scale_d), wq_t, bias);
  KWS_LAUNCH_OK("octize_kernel");
  return KWS_OK;
}
