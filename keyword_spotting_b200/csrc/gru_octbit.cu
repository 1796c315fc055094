// The octbit-rewritten deployment graph (graph_octbit.pb, main.py:357-371): GRU layers whose MatMuls the rewriter
// converts (octbit/octbit_graph.py:218-225: every MatMul that is not in cell_0 -- gates and candidate of the upper
// layers, and the FC) run through OctbitMatMul arithmetic (octbit/octbit_mat_mul_op.cc:90-181) instead of fp32.
//
// The op derives its activation quantiser from the min / max of the WHOLE tensor it is called with.  The reference
// deploys at batch 1, so that range is per stream: per time step for the two GRU MatMuls ([1, 256] inputs: [x_t | h]
// and [x_t | r*h]) and per chunk for the FC ([n, 128]: all frames of the call).  The batched kernels here keep those
// per-stream ranges, i.e. they are S independent copies of the reference's batch-1 graph.
//
//   gru_octbit_layer_kernel : one warp owns 16 streams (rows of mma.sync.m16n8k32 u8 x s8 -> s32) for a whole layer;
//       per step and stream: range of [x_t | h] -> u8 -> gates = octbit(.) + b -> sigmoid; range of [x_t | r*h] -> u8
//       -> candidate = octbit(.) + b -> tanh -> h'.  The unsaturated pair sums come from the tensor cores, the int16
//       saturation of _mm_maddubs_epi16 from a sparse correction over the only pairs that can overflow (same-sign
//       neighbours with |w0|+|w1| >= 129; lists built once per weight at kws_model_set_octbit), and the fp32
//       epilogue is the op's own (octbit_common.cuh).  K = 256 <= 512, so the op's lane-ordered fp32 accumulation
//       equals the exact integer total (octbit.cu).
//   fc_octbit_softmax_kernel: one warp per stream: range over the stream's frames -> u8 -> octbit FC -> + b -> softmax.
#include <cfloat>

#include "common.cuh"
#include "octbit_common.cuh"

namespace kws {

constexpr int kOctTile = 64;            // streams per CTA = tile of the fp32 kernel's [tile][t][unit][64] hand-off
constexpr int kOctWarpStreams = 16;     // rows of one mma
constexpr int kOctCtaWarps = 2;          // warps per CTA: 37.6 KB of shared memory per warp -> three 2-warp CTAs (6 warps) per SM
                                        // instead of one 4-warp CTA; the warps of a tile never talk to each other
constexpr int kOctThreads = 32 * kOctCtaWarps;
constexpr int kOctPartsPerTile = (kOctTile / kOctWarpStreams) / kOctCtaWarps;
constexpr int kOctK = 2 * kHidden;      // [x | h]
constexpr int kOctAStride = kOctK + 4;  // floats per row of the fp32 vector (bank spread, 16-byte aligned)
constexpr int kOctQStride = kOctK + 16; // bytes per row of the u8 vector (conflict-free fragment loads)

struct OctMatDev {
  const signed char* wq;        // [B, K] int8
  const float* obias;           // [B] the op's `bias` attr (127 * column sums)
  float scale;                  // the op's `scale` attr
  const int* cand_count;        // [B]
  const unsigned short* cand;   // [B, K/2] pair indices that can saturate
};

struct GruOctParams {
  long S;
  int n;
  const float* x_tiled;         // [tiles64, n, H, 64] fp32: the layer below (gru.cu hand-off layout)
  float* y_tiled;               // same layout, for the layer above, or null
  float* y_rows;                // [S, n, H] row-major, for the FC, or null
  OctMatDev g, c;               // gates [2H, 2H], candidate [H, 2H]
  const float* bg;              // [2H] fp32 BiasAdd
  const float* bc;              // [H]
  const float* h_in;
  float* h_out;
  const int* seq_len;
  const unsigned char* zero_state;
};

// Warp-level: ranges of the 16 rows of `af`, then their u8 images in `q`.  Lane = (row = lane / 2, half = lane % 2).
__device__ __forceinline__ void quantise_rows(const float* af, unsigned char* q, float* bscale_out, int* signed_out, int lane) {
  const int row = lane >> 1, half = lane & 1;
  const float* src = af + row * kOctAStride + half * kHidden;
  float mn = FLT_MAX, mx = -FLT_MAX;                       // numeric_limits max / lowest (:92-93)
  for (int j = 0; j < kHidden; ++j) {
    const float v = src[j];
    if (v < mn) mn = v;                                    // NaN compares false, as in :96-97
    if (v > mx) mx = v;
  }
  mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, 1));
  mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
  const QuantParams p = quant_from_range(mn, mx);
  if (half == 0) {
    bscale_out[row] = p.bscale;
    signed_out[row] = p.is_signed;
  }
  unsigned* dst = reinterpret_cast<unsigned*>(q + row * kOctQStride + half * kHidden);
  for (int j = 0; j < kHidden; j += 4)
    dst[j >> 2] = quant_one(src[j], p) | (quant_one(src[j + 1], p) << 8) | (quant_one(src[j + 2], p) << 16) |
                  (quant_one(src[j + 3], p) << 24);
}

// sum over the pairs of output `nout` that can saturate of sat16(p) - p, for the u8 row `qrow`
__device__ __forceinline__ int oct_correction(const OctMatDev& m, int nout, const unsigned char* qrow) {
  const int cnt = __ldg(m.cand_count + nout);
  int delta = 0;
  for (int i = 0; i < cnt; ++i) {
    const int kp = __ldg(m.cand + static_cast<long>(nout) * (kOctK / 2) + i);
    const signed char* wr = m.wq + static_cast<long>(nout) * kOctK + 2 * kp;
    const int p = static_cast<int>(qrow[2 * kp]) * __ldg(wr) + static_cast<int>(qrow[2 * kp + 1]) * __ldg(wr + 1);
    delta += sat16(p) - p;
  }
  return delta;
}

// acc[j][e] for 8 n-tiles (64 outputs starting at n0) of matrix m against the warp's 16 u8 rows
__device__ __forceinline__ void oct_mma_chunk(int (&acc)[8][4], const OctMatDev& m, int n0, const unsigned char* q, int lane) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0;
  const unsigned char* q0 = q + g * kOctQStride;
  const unsigned char* q1 = q + (g + 8) * kOctQStride;
#pragma unroll 2
  for (int k0 = 0; k0 < kOctK; k0 += 32) {
    unsigned a[4];
    a[0] = *reinterpret_cast<const unsigned*>(q0 + k0 + 4 * t);
    a[1] = *reinterpret_cast<const unsigned*>(q1 + k0 + 4 * t);
    a[2] = *reinterpret_cast<const unsigned*>(q0 + k0 + 16 + 4 * t);
    a[3] = *reinterpret_cast<const unsigned*>(q1 + k0 + 16 + 4 * t);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const signed char* wr = m.wq + static_cast<long>(n0 + 8 * j + g) * kOctK + k0 + 4 * t;
      const unsigned b0 = __ldg(reinterpret_cast<const unsigned*>(wr));
      const unsigned b1 = __ldg(reinterpret_cast<const unsigned*>(wr + 16));
      mma_u8s8(acc[j], a, b0, b1);
    }
  }
}

__global__ void __launch_bounds__(kOctThreads)
gru_octbit_layer_kernel(const GruOctParams p) {
  extern __shared__ __align__(16) unsigned char smem_oct[];
  const int cta_warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // per-warp regions (a warp never touches another warp's streams: only __syncwarp inside the time loop)
  constexpr size_t kPerWarp = sizeof(float) * kOctWarpStreams * kOctAStride + kOctWarpStreams * kOctQStride +
                              sizeof(float) * 2 * kOctWarpStreams * kHidden + sizeof(float) * kOctWarpStreams +
                              sizeof(int) * 2 * kOctWarpStreams;
  unsigned char* base = smem_oct + cta_warp * kPerWarp;
  float* af = reinterpret_cast<float*>(base);                                 // [16][260]  [x | h] then [x | r*h]
  unsigned char* q = reinterpret_cast<unsigned char*>(af + kOctWarpStreams * kOctAStride);   // [16][272]
  float* hs = reinterpret_cast<float*>(q + kOctWarpStreams * kOctQStride);    // [16][128] fp32 state
  float* us = hs + kOctWarpStreams * kHidden;                                 // [16][128] update gate
  float* bscale = us + kOctWarpStreams * kHidden;                             // [16]
  int* is_signed = reinterpret_cast<int*>(bscale + kOctWarpStreams);          // [16]
  int* lens = is_signed + kOctWarpStreams;                                    // [16]
  const int g = lane >> 2, t4 = lane & 3;
  const long ntiles = (p.S + kOctTile - 1) / kOctTile;

  for (long part = blockIdx.x; part < ntiles * kOctPartsPerTile; part += gridDim.x) {
    const long tile = part / kOctPartsPerTile;
    const int warp = static_cast<int>(part - tile * kOctPartsPerTile) * kOctCtaWarps + cta_warp;   // this warp's 16 streams of the tile
    const long s_warp = tile * kOctTile + warp * kOctWarpStreams;
    // ---- carried state -> hs
    for (int i = lane; i < kOctWarpStreams * kHidden / 4; i += 32) {
      const int r = i / (kHidden / 4), c4 = i - r * (kHidden / 4);
      const long s = s_warp + r;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (s < p.S && !(p.zero_state && p.zero_state[s])) v = *reinterpret_cast<const float4*>(p.h_in + s * kHidden + 4 * c4);
      *reinterpret_cast<float4*>(hs + r * kHidden + 4 * c4) = v;
    }
    if (lane < kOctWarpStreams) {
      const long s = s_warp + lane;
      lens[lane] = s < p.S ? (p.seq_len ? p.seq_len[s] : p.n) : 0;
    }
    __syncwarp();

    for (int t = 0; t < p.n; ++t) {
      // ---- af = [x_t | h]: x from the tiled hand-off (unit-major, 64 streams contiguous)
      {
        const float* xt = p.x_tiled + ((tile * p.n + t) * static_cast<long>(kHidden)) * kOctTile + warp * kOctWarpStreams;
        for (int i = lane; i < kHidden * kOctWarpStreams; i += 32) {
          const int j = i >> 4, r = i & 15;                 // 16 consecutive streams of unit j: 64 contiguous bytes
          af[r * kOctAStride + j] = __ldg(xt + static_cast<long>(j) * kOctTile + r);
        }
        for (int i = lane; i < kOctWarpStreams * kHidden; i += 32) {
          const int r = i >> 7, j = i & 127;
          af[r * kOctAStride + kHidden + j] = hs[r * kHidden + j];
        }
      }
      __syncwarp();
      quantise_rows(af, q, bscale, is_signed, lane);
      __syncwarp();
      // ---- gates: 4 chunks of 64 outputs; outputs 0..127 = r, 128..255 = u
#pragma unroll 1
      for (int ch = 0; ch < 4; ++ch) {
        int acc[8][4];
        oct_mma_chunk(acc, p.g, 64 * ch, q, lane);
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int nout = 64 * ch + 8 * j + 2 * t4 + (e & 1);
            const int r = (e & 2) ? g + 8 : g;
            const int total = acc[j][e] + oct_correction(p.g, nout, q + r * kOctQStride);
            const float val = octbit_epilogue(total, 0, 0, 0, is_signed[r], __ldg(p.g.obias + nout),
                                              __fmul_rn(p.g.scale, bscale[r]));
            const float act = 1.0f / (1.0f + expf(-(val + __ldg(p.bg + nout))));
            if (nout < kHidden) af[r * kOctAStride + kHidden + nout] = act * hs[r * kHidden + nout];   // r (.) h
            else us[r * kHidden + nout - kHidden] = act;
          }
      }
      __syncwarp();
      // ---- candidate on [x_t | r*h] with its OWN range (a separate op call in the reference graph)
      quantise_rows(af, q, bscale, is_signed, lane);
      __syncwarp();
#pragma unroll 1
      for (int ch = 0; ch < 2; ++ch) {
        int acc[8][4];
        oct_mma_chunk(acc, p.c, 64 * ch, q, lane);
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int nout = 64 * ch + 8 * j + 2 * t4 + (e & 1);
            const int r = (e & 2) ? g + 8 : g;
            const int total = acc[j][e] + oct_correction(p.c, nout, q + r * kOctQStride);
            const float val = octbit_epilogue(total, 0, 0, 0, is_signed[r], __ldg(p.c.obias + nout),
                                              __fmul_rn(p.c.scale, bscale[r]));
            const float cand = tanhf(val + __ldg(p.bc + nout));
            const float h = hs[r * kHidden + nout], u = us[r * kHidden + nout];
            const bool live = t < lens[r];
            const float hn = u * h + (1.0f - u) * cand;
            if (live) hs[r * kHidden + nout] = hn;
            // the step's output (zero past the length), parked in the x half of af (x_t is dead now)
            af[r * kOctAStride + nout] = live ? hn : 0.0f;
          }
      }
      __syncwarp();
      // ---- outputs
      if (p.y_tiled) {
        float* yt = p.y_tiled + ((tile * p.n + t) * static_cast<long>(kHidden)) * kOctTile + warp * kOctWarpStreams;
        for (int i = lane; i < kHidden * kOctWarpStreams; i += 32) {
          const int j = i >> 4, r = i & 15;
          yt[static_cast<long>(j) * kOctTile + r] = af[r * kOctAStride + j];
        }
      }
      if (p.y_rows) {
        for (int i = lane; i < kOctWarpStreams * kHidden / 4; i += 32) {
          const int r = i / (kHidden / 4), c4 = i - r * (kHidden / 4);
          const long s = s_warp + r;
          if (s < p.S)
            *reinterpret_cast<float4*>(p.y_rows + (s * p.n + t) * kHidden + 4 * c4) =
                *reinterpret_cast<const float4*>(af + r * kOctAStride + 4 * c4);
        }
      }
      __syncwarp();
    }
    // ---- final state
    for (int i = lane; i < kOctWarpStreams * kHidden / 4; i += 32) {
      const int r = i / (kHidden / 4), c4 = i - r * (kHidden / 4);
      const long s = s_warp + r;
      if (s < p.S) *reinterpret_cast<float4*>(p.h_out + s * kHidden + 4 * c4) = *reinterpret_cast<const float4*>(hs + r * kHidden + 4 * c4);
    }
    __syncwarp();
  }
}

static size_t gru_octbit_smem_bytes() {
  const size_t per_warp = sizeof(float) * kOctWarpStreams * kOctAStride + kOctWarpStreams * kOctQStride +
                          sizeof(float) * 2 * kOctWarpStreams * kHidden + sizeof(float) * kOctWarpStreams +
                          sizeof(int) * 2 * kOctWarpStreams;
  return per_warp * kOctCtaWarps;
}

// FC + softmax on the last layer's outputs y [S, n, H]: one warp per stream.
//   octbit FC: ONE op call per stream and chunk (inference2 flattens all frames of the batch-1 call,
//   models/rnn_ctc.py:268-277): range over the stream's `len` frames, K = 128, every pair formed and saturated.
//   fp32 FC (the graph's FC left unconverted): plain fp32 dot products.
struct FcOctParams {
  long S;
  int n, C;
  const float* y;               // [S, n, H]
  const int* seq_len;
  int octbit;
  OctMatDev fc;                 // [C, H]
  const float* fc_w;            // [H, C] fp32 (when !octbit)
  const float* fc_b;            // [C]
  float* probs;
  float* logits;
};

__global__ void __launch_bounds__(128)
fc_octbit_softmax_kernel(const FcOctParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long s = blockIdx.x * 4L + warp;
  if (s >= p.S) return;
  const float* ys = p.y + s * p.n * static_cast<long>(kHidden);
  const int len = p.seq_len ? min(p.seq_len[s], p.n) : p.n;
  QuantParams qp;
  qp.bscale = 0.0f;
  qp.offset = 0.0f;
  qp.is_signed = 0;
  if (p.octbit) {
    float mn = FLT_MAX, mx = -FLT_MAX;
    for (int i = lane; i < len * kHidden; i += 32) {
      const float v = ys[i];
      if (v < mn) mn = v;
      if (v > mx) mx = v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    qp = quant_from_range(mn, mx);
  }
  for (int t = lane; t < p.n; t += 32) {                   // lane = frame
    const float* row = ys + static_cast<long>(t) * kHidden;
    float lg[kMaxClasses];
    if (p.octbit) {
      int tot[kMaxClasses];
      for (int c = 0; c < p.C; ++c) tot[c] = 0;
      for (int k = 0; k < kHidden; k += 2) {
        const int q0 = static_cast<int>(quant_one(row[k], qp)), q1 = static_cast<int>(quant_one(row[k + 1], qp));
        for (int c = 0; c < p.C; ++c) {
          const signed char* wr = p.fc.wq + c * kHidden + k;
          tot[c] += sat16(q0 * __ldg(wr) + q1 * __ldg(wr + 1));
        }
      }
      const float scale = __fmul_rn(p.fc.scale, qp.bscale);
      for (int c = 0; c < p.C; ++c)
        lg[c] = octbit_epilogue(tot[c], 0, 0, 0, qp.is_signed, __ldg(p.fc.obias + c), scale) + __ldg(p.fc_b + c);
    } else {
      for (int c = 0; c < p.C; ++c) lg[c] = 0.0f;
      for (int k = 0; k < kHidden; ++k) {
        const float v = row[k];
        for (int c = 0; c < p.C; ++c) lg[c] = fmaf(v, __ldg(p.fc_w + k * p.C + c), lg[c]);
      }
      for (int c = 0; c < p.C; ++c) lg[c] += __ldg(p.fc_b + c);
    }
    float mxl = -INFINITY;
    for (int c = 0; c < p.C; ++c) mxl = fmaxf(mxl, lg[c]);
    float e[kMaxClasses], sum = 0.0f;
    for (int c = 0; c < p.C; ++c) {
      e[c] = expf(lg[c] - mxl);
      sum += e[c];
    }
    float* pr = p.probs + (s * p.n + t) * p.C;
    for (int c = 0; c < p.C; ++c) pr[c] = e[c] / sum;
    if (p.logits) {
      float* lo = p.logits + (s * p.n + t) * p.C;
      for (int c = 0; c < p.C; ++c) lo[c] = lg[c];
    }
  }
}

static void free_oct(OctbitMatrix& o) {
  cudaFree(o.wq);
  cudaFree(o.obias);
  cudaFree(o.cand_count);
  cudaFree(o.cand);
  o = OctbitMatrix();
}

void free_octbit(kws_model* m) {
  for (int l = 0; l < kMaxLayers; ++l) {
    free_oct(m->oct_gates[l]);
    free_oct(m->oct_cand[l]);
  }
  free_oct(m->oct_fc);
  cudaFree(m->oct_y_rows);
  m->oct_y_rows = nullptr;
  m->oct_y_bytes = 0;
  m->octbit = false;
}

static int upload_oct(OctbitMatrix* dst, const int8_t* wq, const float* obias, float scale, int B, int K) {
  KWS_REQUIRE(scale > 0.0f, "scale has to be positive");                   // octbit_mat_mul_op.cc:45-46
  KWS_REQUIRE(K % 64 == 0, "we need to be 16 aligned. K=%d", K);           // :65-67
  dst->B = B;
  dst->K = K;
  dst->scale = scale;
  KWS_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&dst->wq), static_cast<size_t>(B) * K));
  KWS_CUDA_OK(cudaMemcpy(dst->wq, wq, static_cast<size_t>(B) * K, cudaMemcpyHostToDevice));
  KWS_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&dst->obias), sizeof(float) * B));
  KWS_CUDA_OK(cudaMemcpy(dst->obias, obias, sizeof(float) * B, cudaMemcpyHostToDevice));
  KWS_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&dst->cand_count), sizeof(int) * B));
  KWS_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&dst->cand), sizeof(unsigned short) * static_cast<size_t>(B) * (K / 2)));
  // the list order is the atomics' and differs from run to run; the correction is an integer sum over the list
  KWS_CUDA_OK(cudaMemset(dst->cand_count, 0, sizeof(int) * B));
  octbit_find_candidates_kernel<<<static_cast<unsigned>(ceil_div(static_cast<int64_t>(B) * (K / 2), 256)), 256>>>(
      dst->wq, B, K, dst->cand_count, dst->cand);
  KWS_LAUNCH_OK("octbit_find_candidates_kernel");
  KWS_CUDA_OK(cudaDeviceSynchronize());
  return KWS_OK;
}

static OctMatDev dev_view(const OctbitMatrix& o) {
  OctMatDev d;
  d.wq = o.wq;
  d.obias = o.obias;
  d.scale = o.scale;
  d.cand_count = o.cand_count;
  d.cand = o.cand;
  return d;
}

int launch_octbit_layer(kws_model* m, const GruArgs& a, int l, const float* x_tiled, float* y_tiled, float* y_rows,
                        cudaStream_t st) {
  GruOctParams p;
  p.S = a.S;
  p.n = a.n;
  p.x_tiled = x_tiled;
  p.y_tiled = y_tiled;
  p.y_rows = y_rows;
  p.g = dev_view(m->oct_gates[l]);
  p.c = dev_view(m->oct_cand[l]);
  p.bg = m->layer[l].gates_bias;
  p.bc = m->layer[l].cand_bias;
  p.h_in = a.state_in + static_cast<long>(l) * a.S * kHidden;
  p.h_out = a.state_out + static_cast<long>(l) * a.S * kHidden;
  p.seq_len = a.seq_len;
  p.zero_state = a.zero_state;
  const size_t smem = gru_octbit_smem_bytes();
  KWS_CUDA_OK(cudaFuncSetAttribute(gru_octbit_layer_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const long parts = ceil_div(a.S, kOctTile) * kOctPartsPerTile;
  const long blocks = parts < 3L * sm_count() ? parts : 3L * sm_count();
  gru_octbit_layer_kernel<<<static_cast<unsigned>(blocks), kOctThreads, smem, st>>>(p);
  KWS_LAUNCH_OK("gru_octbit_layer_kernel");
  return KWS_OK;
}

int launch_octbit_fc(kws_model* m, const GruArgs& a, const float* y_rows, cudaStream_t st) {
  FcOctParams f;
  f.S = a.S;
  f.n = a.n;
  f.C = m->cfg.num_classes;
  f.y = y_rows;
  f.seq_len = a.seq_len;
  f.octbit = m->oct_fc.wq != nullptr;
  f.fc = dev_view(m->oct_fc);
  f.fc_w = m->fc_w;
  f.fc_b = m->fc_b;
  f.probs = a.probs;
  f.logits = a.logits;
  fc_octbit_softmax_kernel<<<static_cast<unsigned>(ceil_div(a.S, 4)), 128, 0, st>>>(f);
  KWS_LAUNCH_OK("fc_octbit_softmax_kernel");
  return KWS_OK;
}

}  // namespace kws

using namespace kws;

extern "C" int kws_model_set_octbit(kws_model* m, const kws_octbit_weights* w) {
  clear_error();
  KWS_REQUIRE(m != nullptr, "model is NULL");
  KWS_CUDA_OK(cudaSetDevice(m->device));
  KWS_CUDA_OK(cudaDeviceSynchronize());
  free_octbit(m);
  if (!w) return KWS_OK;                                    // back to the float graph
  const int L = m->cfg.num_layers, C = m->cfg.num_classes;
  bool any = false;
  for (int l = 0; l < L; ++l) {
    const bool has_g = w->gates_wq[l] != nullptr, has_c = w->cand_wq[l] != nullptr;
    KWS_REQUIRE(has_g == has_c, "layer %d: gates and candidate must both be octbit or both float", l);
    if (!has_g) continue;
    KWS_REQUIRE(l >= 1 && m->layer[l].in_dim == kHidden,
                "layer %d: only layers fed by a GRU layer can be octbit (the rewriter skips cell_0, octbit_graph.py:218-225)", l);
    KWS_REQUIRE(w->gates_obias[l] && w->cand_obias[l], "layer %d: NULL octbit bias", l);
    int rc = upload_oct(&m->oct_gates[l], w->gates_wq[l], w->gates_obias[l], w->gates_scale[l], 2 * kHidden, 2 * kHidden);
    if (rc == KWS_OK) rc = upload_oct(&m->oct_cand[l], w->cand_wq[l], w->cand_obias[l], w->cand_scale[l], kHidden, 2 * kHidden);
    if (rc != KWS_OK) {
      const std::string msg = kws_last_error();
      free_octbit(m);
      set_error("%s", msg.c_str());
      return rc;
    }
    any = true;
  }
  if (w->fc_wq) {
    KWS_REQUIRE(w->fc_obias != nullptr, "NULL octbit FC bias");
    const int rc = upload_oct(&m->oct_fc, w->fc_wq, w->fc_obias, w->fc_scale, C, kHidden);
    if (rc != KWS_OK) {
      const std::string msg = kws_last_error();
      free_octbit(m);
      set_error("%s", msg.c_str());
      return rc;
    }
    any = true;
  }
  m->octbit = any;
  return KWS_OK;
}

extern "C" int kws_model_is_octbit(const kws_model* m) { return m && m->octbit ? 1 : 0; }
