// Shared pieces of the octbit back ends: workspace header, activation quantiser and the fp32 epilogue, all
// bit-exact restatements of OctbitMatMulOp::Compute (octbit/octbit_mat_mul_op.cc:90-181).
#pragma once

#include "common.cuh"

namespace kws {

struct OctbitHeader {        // first 256 bytes of the workspace
  unsigned enc_min;          // order-preserving encodings of the running min / max
  unsigned enc_max;
  unsigned pad[62];
};

__device__ __forceinline__ unsigned enc_float(float f) {
  unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float dec_float(unsigned e) {
  unsigned u = (e & 0x80000000u) ? (e & 0x7fffffffu) : ~e;
  return __uint_as_float(u);
}

struct QuantParams {
  float bscale;
  float offset;     // 127 (signed) or 0
  int is_signed;
};

// the quantiser of a tensor whose elements span [mn, mx]   (:90-124)
__device__ __forceinline__ QuantParams quant_from_range(float mn, float mx) {
  QuantParams p;
  p.is_signed = mn < 0.0f;
  if (p.is_signed) {
    p.bscale = __fdiv_rn(fmaxf(-mn, mx), 127.0f);
    p.offset = 127.0f;
  } else {
    p.bscale = __fdiv_rn(mx, 254.0f);
    p.offset = 0.0f;
  }
  return p;
}
__device__ __forceinline__ QuantParams quant_params(const OctbitHeader* h) {
  return quant_from_range(dec_float(h->enc_min), dec_float(h->enc_max));
}

__device__ __forceinline__ unsigned quant_one(float x, const QuantParams& p) {
  if (p.bscale == 0.0f) return 0u;                       // 0/0: undefined in the reference
  const float r = roundf(__fdiv_rn(x, p.bscale));        // C round(): half away from zero
  return static_cast<unsigned>(static_cast<int>(r + p.offset)) & 0xffu;
}

__device__ __forceinline__ int sat16(int v) { return max(-32768, min(32767, v)); }

__device__ __forceinline__ float octbit_epilogue(int l0, int l1, int l2, int l3, int is_signed,
                                                 float bias, float scale) {
  float o = 0.0f;                                   // output(batch,i) = 0          (:127-131)
  o = __fadd_rn(o, static_cast<float>(l0));         // += val[m], m = 0..3          (:172-175)
  o = __fadd_rn(o, static_cast<float>(l1));
  o = __fadd_rn(o, static_cast<float>(l2));
  o = __fadd_rn(o, static_cast<float>(l3));
  if (is_signed) o = __fsub_rn(o, bias);            // -= biasvec(i)                (:176-178)
  return __fmul_rn(o, scale);                       // *= scale                     (:179)
}

__device__ __forceinline__ void mma_u8s8(int (&c)[4], const unsigned (&a)[4], unsigned b0, unsigned b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
      "{%0,%1,%2,%3};\n"
      : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// Saturation candidates (octbit.cu): the pairs of weight row n that can overflow int16 for some u8 row, appended to
// cand[n * K/2 ..] in any order; cand_count[n] counts them and must be zero before the launch.
__global__ void __launch_bounds__(256)
octbit_find_candidates_kernel(const signed char* __restrict__ w, int B, int K, int* __restrict__ cand_count,
                              unsigned short* __restrict__ cand);

// tensor-core (tcgen05 kind::i8) back end with the quantiser fused in, octbit_tc.cu
bool octbit_tc_supported(int64_t A, int64_t B, int64_t K);
int launch_octbit_tc(const float* x, const int8_t* w, const float* bias, float scale_attr, int64_t A, int64_t B, int64_t K,
                     const OctbitHeader* hdr, const int* cand_count, const unsigned short* cand, float* out,
                     cudaStream_t st);

}  // namespace kws
