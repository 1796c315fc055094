// attention_ctc deployment forward pass (BASELINE config 5; SURVEY.md 8f row 2) -- the consumer of the K6
// positional-encoding op.
//
// Reference: models/attention_ctc.py:73-128 (inference), :28-58 (self_attention), :61-70 (feed_forward),
// :215-274 (DeployModel).  Per batch of utterances, on mel frames [B, T, M] of which utterance b has lens[b] valid:
//   combine_frame=2 folding with the reference's padding rule (T' = T/2 + 1)       :77-90
//   input_linear_trans (1x1 conv = dense + bias) + positional_encoding(T', N)       :92-98
//   3 x { qkv dense, 8-head softmax(q k^T / sqrt(16)) v over ALL T' keys (no mask),
//         layer_norm(att + x), relu FFN 128->512->128, layer_norm(ffn + y) }         :100-120
//   output_linear_trans (+ relu when config.use_relu) and softmax                    :122-127, :272
// tf.contrib.layers.layer_norm of that TensorFlow era normalises over all non-batch axes of [B, T', N]
// (one mean/variance per utterance), gamma/beta per channel, epsilon 1e-12.
//
// Variable-length batches: every utterance is computed exactly as the graph computes it alone on its own lens[b] frames
// (batch-1 sess.run): T'_b = att_frames(lens[b]) rows folded with zeros after frame lens[b], positions 0 .. T'_b - 1,
// keys 0 .. T'_b - 1 only, layer-norm moments over T'_b x N; output rows T'_b .. T' - 1 are zero.  Rows keep the stride
// T' of the longest utterance; each kernel reads its utterance's T'_b through AttLens (common.cuh) and never reads mel
// frames at or past lens[b] or activation rows at or past T'_b.  Because every kernel does per utterance (attention
// core, layer norm) or per row (dense, output) the same arithmetic as at T' = T'_b, the valid rows are bit-identical to
// a call on that utterance alone.
//
// Dense layers: tcgen05 with fp16 hi/lo operand splits, fp32-grade (attention_tc.cu); the fp32 FFMA GEMM below remains for
// shapes that kernel does not take.  Attention itself: one thread per query, online softmax, K/V blocks staged in shared
// memory (fp32 FFMA); per-utterance fused add + layer-norm.  The work is 0.7 GFLOP per 8 s utterance.
#include <cmath>
#include <vector>

#include "common.cuh"

struct kws_attention {
  kws_attention_config cfg;
  int device = 0;
  float *w_in = nullptr, *b_in = nullptr, *w_out = nullptr, *b_out = nullptr;
  struct Layer {
    float *w_qkv = nullptr, *b_qkv = nullptr, *ln1_g = nullptr, *ln1_b = nullptr;
    float *w_ff1 = nullptr, *b_ff1 = nullptr, *w_ff2 = nullptr, *b_ff2 = nullptr, *ln2_g = nullptr, *ln2_b = nullptr;
  } layer[8];
  // the dense layers' weights as pre-split fp16 tensor-core operands (attention_tc.cu); null -> the FFMA kernel
  struct Packed {
    unsigned char* w = nullptr;
    int nchunks = 0;
  } p_in, p_qkv[8], p_ff1[8], p_ff2[8];
  float* pe = nullptr;          // [pe_rows, N] from the K6 kernel
  int pe_rows = 0;
  float* scratch = nullptr;     // xin | x | y | att | big, each segment padded to 32 floats
  size_t scratch_floats = 0;
};

namespace kws {

bool att_linear_tc_supported(int K, int N);                                                   // attention_tc.cu
int att_pack_linear(const float* W, int K, int N, unsigned char** out, int* nchunks_out);
int launch_att_linear_tc(const float* A, const unsigned char* wpack, int nchunks, const float* bias, const float* pe, int Tp,
                         AttLens lens, long rows, int K, int N, bool relu, bool add_pe, float* Y, cudaStream_t st);
bool att_core_tc_supported(int Tp, int heads, int hidden);
int launch_att_core_tc(const float* qkv, long B, int Tp, int heads, AttLens lens, float* out, cudaStream_t st);

constexpr int kAttHidden = 128;
constexpr int kAttHeadDim = 16;

// ---- fold `combine` frames into one row with the reference's zero padding (:77-90) after the utterance's last frame
// (rows at or past T'_b come out zero: their first frame lies past lens[b])
__global__ void att_combine_kernel(const float* __restrict__ mel, long B, int T, int M, int combine, int Tp, AttLens lens,
                                   float* __restrict__ out) {
  const long idx = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  const int K = M * combine;
  const long total = B * Tp * K;
  if (idx >= total) return;
  const int j = static_cast<int>(idx % K);
  const long row = idx / K;
  const int tp = static_cast<int>(row % Tp);
  const long b = row / Tp;
  const int f = tp * combine + j / M;
  out[idx] = f < lens.frames_in(b) ? mel[(b * T + f) * M + j % M] : 0.0f;
}

// ---- Y[r, n] = act(sum_k A[r,k] W[k,n] + bias[n]) (+ pe[r % Tp, n]);  64x64 tile, 256 threads x (4x4); a tile of
// padding rows only (at or past their utterances' T'_b) does nothing
template <bool kRelu, bool kAddPe>
__global__ void __launch_bounds__(256)
att_linear_kernel(const float* __restrict__ A, const float* __restrict__ W, const float* __restrict__ bias,
                  const float* __restrict__ pe, int Tp, AttLens lens, long rows, int K, int N, float* __restrict__ Y) {
  if (!lens.tile_live(Tp, rows, blockIdx.x * 64L, 64)) return;
  __shared__ float sA[16][64 + 4];
  __shared__ float sW[16][64];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;          // 16 x 16 threads
  const long r0 = blockIdx.x * 64L;
  const int n0 = blockIdx.y * 64;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += 16) {
    for (int i = threadIdx.x; i < 64 * 16; i += 256) {             // A tile, transposed into [k][row]
      const int r = i >> 4, k = i & 15;
      const long gr = r0 + r;
      sA[k][r] = (gr < rows && k0 + k < K) ? A[gr * K + k0 + k] : 0.0f;
    }
    for (int i = threadIdx.x; i < 16 * 64; i += 256) {
      const int k = i >> 6, n = i & 63;
      sW[k][n] = (k0 + k < K && n0 + n < N) ? W[static_cast<long>(k0 + k) * N + n0 + n] : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      float a[4], w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = sA[k][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) w[j] = sW[k][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long r = r0 + ty * 4 + i;
    if (r >= rows) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = acc[i][j] + bias[n];
      if (kRelu) v = fmaxf(v, 0.0f);
      if (kAddPe) v += pe[static_cast<long>(r % Tp) * N + n];
      Y[r * N + n] = v;
    }
  }
}

// ---- multi-head attention: one thread per query row, K/V blocks of 128 keys in shared memory, online softmax over the
// utterance's T'_b keys (Tp is the row stride); utterances with T'_b <= skip_upto are left to the tensor-core core
__global__ void __launch_bounds__(128)
att_attention_kernel(const float* __restrict__ qkv, int Tp, int heads, AttLens lens, int skip_upto,
                     float* __restrict__ out) {
  __shared__ float sK[128][kAttHeadDim];
  __shared__ float sV[128][kAttHeadDim];
  const int N = heads * kAttHeadDim;
  const int h = blockIdx.y;
  const long b = blockIdx.z;
  const int Tb = lens.rows_of(b);
  if (Tb <= skip_upto || blockIdx.x * 128 >= Tb) return;
  const int i = blockIdx.x * 128 + threadIdx.x;
  const float* base = qkv + b * Tp * 3L * N;
  const float scale = rsqrtf(static_cast<float>(kAttHeadDim)) * 1.4426950408889634f;   // 1/sqrt(d), in log2 units
  float q[kAttHeadDim], o[kAttHeadDim];
#pragma unroll
  for (int d = 0; d < kAttHeadDim; ++d) {
    q[d] = i < Tb ? base[static_cast<long>(i) * 3 * N + h * kAttHeadDim + d] * scale : 0.0f;
    o[d] = 0.0f;
  }
  float m = -INFINITY, l = 0.0f;
  for (int j0 = 0; j0 < Tb; j0 += 128) {
    const int j = j0 + threadIdx.x;
    if (j < Tb) {
      const float4* kp = reinterpret_cast<const float4*>(base + static_cast<long>(j) * 3 * N + N + h * kAttHeadDim);
      const float4* vp = reinterpret_cast<const float4*>(base + static_cast<long>(j) * 3 * N + 2 * N + h * kAttHeadDim);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        reinterpret_cast<float4*>(sK[threadIdx.x])[c] = kp[c];
        reinterpret_cast<float4*>(sV[threadIdx.x])[c] = vp[c];
      }
    }
    __syncthreads();
    const int nk = Tb - j0 < 128 ? Tb - j0 : 128;
    for (int jj = 0; jj < nk; ++jj) {
      float s = 0.0f;
#pragma unroll
      for (int d = 0; d < kAttHeadDim; ++d) s = fmaf(q[d], sK[jj][d], s);
      if (s > m) {                                   // rescale only when the running maximum moves
        const float c = exp2f(m - s);
        l *= c;
#pragma unroll
        for (int d = 0; d < kAttHeadDim; ++d) o[d] *= c;
        m = s;
      }
      const float p = exp2f(s - m);
      l += p;
#pragma unroll
      for (int d = 0; d < kAttHeadDim; ++d) o[d] = fmaf(p, sV[jj][d], o[d]);
    }
    __syncthreads();
  }
  if (i < Tb) {
    const float inv = 1.0f / l;
    float* dst = out + (b * Tp + i) * N + h * kAttHeadDim;
#pragma unroll
    for (int d = 0; d < kAttHeadDim; ++d) dst[d] = o[d] * inv;
  }
}

// ---- y = layer_norm(a + b) over all T'_b * N elements of one utterance, per-channel gamma/beta; rows at or past T'_b are
// neither read nor written.  The reduction order depends on T'_b only, not on the row stride Tp nor on in_smem.
__device__ __forceinline__ float block_sum(float v, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[w] = v;
  __syncthreads();
  float t = threadIdx.x < nw ? red[threadIdx.x] : 0.0f;
  if (threadIdx.x < 32) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) red[0] = t;
  }
  __syncthreads();
  return red[0];
}

__global__ void __launch_bounds__(1024)
att_add_layernorm_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ gamma,
                         const float* __restrict__ beta, int Tp, AttLens lens, int N, int in_smem, float* __restrict__ y) {
  // the utterance's a + b is kept in shared memory when it fits (T' * N <= 51,200 floats: 8 s at config 5), so a and b
  // are read from HBM once and the mean / variance / output passes run out of shared memory; N % 4 == 0
  extern __shared__ __align__(16) float sx[];
  __shared__ float red[32];
  const long base = blockIdx.x * static_cast<long>(Tp) * N;
  const int n = lens.rows_of(blockIdx.x) * N, n4 = n >> 2;
  const float4* a4 = reinterpret_cast<const float4*>(a + base);
  const float4* b4 = reinterpret_cast<const float4*>(b + base);
  float4* s4 = reinterpret_cast<float4*>(sx);
  float s = 0.0f;
  for (int i = threadIdx.x; i < n4; i += blockDim.x) {
    const float4 u = __ldg(a4 + i), w = __ldg(b4 + i);
    const float4 t = make_float4(u.x + w.x, u.y + w.y, u.z + w.z, u.w + w.w);
    if (in_smem) s4[i] = t;
    s += (t.x + t.y) + (t.z + t.w);
  }
  const float mean = block_sum(s, red) / n;
  float v = 0.0f;
  for (int i = threadIdx.x; i < n4; i += blockDim.x) {
    float4 t;
    if (in_smem) {
      t = s4[i];
    } else {
      const float4 u = __ldg(a4 + i), w = __ldg(b4 + i);
      t = make_float4(u.x + w.x, u.y + w.y, u.z + w.z, u.w + w.w);
    }
    const float d0 = t.x - mean, d1 = t.y - mean, d2 = t.z - mean, d3 = t.w - mean;
    v = fmaf(d0, d0, v); v = fmaf(d1, d1, v); v = fmaf(d2, d2, v); v = fmaf(d3, d3, v);
  }
  const float var = block_sum(v, red) / n;
  const float inv = 1.0f / sqrtf(var + 1e-12f);
  float4* y4 = reinterpret_cast<float4*>(y + base);
  const int nq = N >> 2;
  for (int i = threadIdx.x; i < n4; i += blockDim.x) {
    float4 t;
    if (in_smem) {
      t = s4[i];
    } else {
      const float4 u = __ldg(a4 + i), w = __ldg(b4 + i);
      t = make_float4(u.x + w.x, u.y + w.y, u.z + w.z, u.w + w.w);
    }
    const int c = (i % nq) << 2;
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c)), be = __ldg(reinterpret_cast<const float4*>(beta + c));
    y4[i] = make_float4((t.x - mean) * inv * g.x + be.x, (t.y - mean) * inv * g.y + be.y, (t.z - mean) * inv * g.z + be.z,
                        (t.w - mean) * inv * g.w + be.w);
  }
}

// ---- output_linear_trans (+relu) + softmax: one thread per row; rows at or past T'_b are written as zeros
__global__ void __launch_bounds__(128)
att_output_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias, long rows,
                  int Tp, AttLens lens, int N, int C, int use_relu, float* __restrict__ probs, float* __restrict__ logits) {
  extern __shared__ float sw[];                       // [N][C] + [C]
  const long r = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  const bool pad = lens.lens && r < rows && r % Tp >= lens.rows_of(r / Tp);   // a row at or past T'_b
  if (pad) {
    for (int c = 0; c < C; ++c) {
      probs[r * C + c] = 0.0f;
      if (logits) logits[r * C + c] = 0.0f;
    }
  }
  for (int i = threadIdx.x; i < N * C; i += blockDim.x) sw[i] = w[i];
  for (int i = threadIdx.x; i < C; i += blockDim.x) sw[N * C + i] = bias[i];
  __syncthreads();
  if (r >= rows || pad) return;
  float acc[kMaxClasses];
  for (int c = 0; c < C; ++c) acc[c] = sw[N * C + c];
  const float4* xr = reinterpret_cast<const float4*>(x + r * N);
  for (int k4 = 0; k4 < N / 4; ++k4) {
    const float4 v = xr[k4];
    const float xs[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e)
      for (int c = 0; c < C; ++c) acc[c] = fmaf(xs[e], sw[(4 * k4 + e) * C + c], acc[c]);
  }
  float mx = -INFINITY;
  for (int c = 0; c < C; ++c) {
    if (use_relu) acc[c] = fmaxf(acc[c], 0.0f);
    mx = fmaxf(mx, acc[c]);
  }
  float sum = 0.0f, e[kMaxClasses];
  for (int c = 0; c < C; ++c) {
    e[c] = expf(acc[c] - mx);
    sum += e[c];
  }
  for (int c = 0; c < C; ++c) {
    probs[r * C + c] = e[c] / sum;
    if (logits) logits[r * C + c] = acc[c];
  }
}

template <typename T>
static int att_upload(T** dst, const T* host, size_t n) {
  *dst = nullptr;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(dst), sizeof(T) * (n ? n : 1));
  if (e != cudaSuccess) return fail(KWS_ERR_ALLOC, "cudaMalloc(%zu) failed: %s", sizeof(T) * n, cudaGetErrorString(e));
  KWS_CUDA_OK(cudaMemcpy(*dst, host, sizeof(T) * n, cudaMemcpyHostToDevice));
  return KWS_OK;
}

static void att_free(kws_attention* m) {
  if (!m) return;
  cudaFree(m->w_in); cudaFree(m->b_in); cudaFree(m->w_out); cudaFree(m->b_out);
  for (auto& l : m->layer) {
    cudaFree(l.w_qkv); cudaFree(l.b_qkv); cudaFree(l.ln1_g); cudaFree(l.ln1_b); cudaFree(l.w_ff1);
    cudaFree(l.b_ff1); cudaFree(l.w_ff2); cudaFree(l.b_ff2); cudaFree(l.ln2_g); cudaFree(l.ln2_b);
  }
  cudaFree(m->p_in.w);
  for (int l = 0; l < 8; ++l) {
    cudaFree(m->p_qkv[l].w);
    cudaFree(m->p_ff1[l].w);
    cudaFree(m->p_ff2[l].w);
  }
  cudaFree(m->pe);
  cudaFree(m->scratch);
  delete m;
}

template <bool R, bool P>
static int att_linear(const float* A, const float* W, const kws_attention::Packed& pk, const float* bias, const float* pe, int Tp,
                      AttLens lens, long rows, int K, int N, float* Y, cudaStream_t st) {
  if (pk.w) return launch_att_linear_tc(A, pk.w, pk.nchunks, bias, pe, Tp, lens, rows, K, N, R, P, Y, st);   // tcgen05, fp32-grade
  dim3 grid(static_cast<unsigned>(ceil_div(rows, 64)), static_cast<unsigned>(ceil_div(N, 64)));
  att_linear_kernel<R, P><<<grid, 256, 0, st>>>(A, W, bias, pe, Tp, lens, rows, K, N, Y);
  KWS_LAUNCH_OK("att_linear_kernel");
  return KWS_OK;
}

static int att_core_ffma(const float* qkv, long B, int Tp, int heads, AttLens lens, int skip_upto, float* out, cudaStream_t st) {
  dim3 ga(static_cast<unsigned>(ceil_div(Tp, 128)), static_cast<unsigned>(heads), static_cast<unsigned>(B));
  att_attention_kernel<<<ga, 128, 0, st>>>(qkv, Tp, heads, lens, skip_upto, out);
  KWS_LAUNCH_OK("att_attention_kernel");
  return KWS_OK;
}

// the attention core of one layer.  Every utterance goes to the core a call on it alone would use: the tensor cores when
// T'_b <= 400, the FFMA kernel otherwise.  With T' <= 400 that is the tcgen05 core alone; past it, with lengths, both
// kernels run and each returns at once for the other's utterances.
static int att_core(const float* qkv, long B, int Tp, int heads, AttLens lens, float* out, cudaStream_t st) {
  if (att_core_tc_supported(Tp, heads, heads * kAttHeadDim)) return launch_att_core_tc(qkv, B, Tp, heads, lens, out, st);
  if (lens.lens) {
    const int rc = launch_att_core_tc(qkv, B, Tp, heads, lens, out, st);
    if (rc != KWS_OK) return rc;
    return att_core_ffma(qkv, B, Tp, heads, lens, kAttCoreTcMaxKeys, out, st);
  }
  return att_core_ffma(qkv, B, Tp, heads, lens, 0, out, st);
}

constexpr int kLnSmemBytes = 200 * 1024;       // the layer norm keeps a + b in shared memory up to this size

}  // namespace kws

using namespace kws;

extern "C" int kws_attention_create(const kws_attention_config* cfg, const kws_attention_weights* w, int device,
                                    kws_attention** out) {
  clear_error();
  KWS_REQUIRE(cfg && w && out, "NULL argument");
  *out = nullptr;
  KWS_REQUIRE(cfg->hidden == kAttHidden, "hidden_size must be %d (config/attention_config.py:85)", kAttHidden);
  KWS_REQUIRE(cfg->heads >= 1 && cfg->hidden == cfg->heads * kAttHeadDim, "the attention kernel is built for head size %d", kAttHeadDim);
  KWS_REQUIRE(cfg->num_layers >= 1 && cfg->num_layers <= 8, "num_layers must be in [1, 8]");
  KWS_REQUIRE(cfg->num_classes >= 2 && cfg->num_classes <= kMaxClasses, "num_classes must be in [2, %d]", kMaxClasses);
  KWS_REQUIRE(cfg->n_mel >= 1 && cfg->combine_frame >= 1 && cfg->ffn >= 1, "bad sizes");
  KWS_REQUIRE(w->w_in && w->b_in && w->w_out && w->b_out, "NULL weight pointer");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0)
    return fail(KWS_ERR_CUDA, "no CUDA device available (%s); libkws_b200 has no CPU fallback",
                e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
  KWS_REQUIRE(device >= 0 && device < ndev, "device %d out of range [0, %d)", device, ndev);
  KWS_CUDA_OK(cudaSetDevice(device));
  kws_attention* m = new kws_attention();
  m->cfg = *cfg;
  m->device = device;
  const int N = cfg->hidden, F = cfg->ffn, C = cfg->num_classes, Kin = cfg->n_mel * cfg->combine_frame;
  int rc = att_upload(&m->w_in, w->w_in, static_cast<size_t>(Kin) * N);
  if (rc == KWS_OK) rc = att_upload(&m->b_in, w->b_in, N);
  for (int l = 0; l < cfg->num_layers && rc == KWS_OK; ++l) {
    if (!(w->w_qkv[l] && w->b_qkv[l] && w->ln1_g[l] && w->ln1_b[l] && w->w_ff1[l] && w->b_ff1[l] && w->w_ff2[l] &&
          w->b_ff2[l] && w->ln2_g[l] && w->ln2_b[l])) {
      att_free(m);
      return fail(KWS_ERR_INVALID_ARGUMENT, "NULL weight pointer for layer %d", l);
    }
    auto& L = m->layer[l];
    rc = att_upload(&L.w_qkv, w->w_qkv[l], static_cast<size_t>(N) * 3 * N);
    if (rc == KWS_OK) rc = att_upload(&L.b_qkv, w->b_qkv[l], 3 * N);
    if (rc == KWS_OK) rc = att_upload(&L.ln1_g, w->ln1_g[l], N);
    if (rc == KWS_OK) rc = att_upload(&L.ln1_b, w->ln1_b[l], N);
    if (rc == KWS_OK) rc = att_upload(&L.w_ff1, w->w_ff1[l], static_cast<size_t>(N) * F);
    if (rc == KWS_OK) rc = att_upload(&L.b_ff1, w->b_ff1[l], F);
    if (rc == KWS_OK) rc = att_upload(&L.w_ff2, w->w_ff2[l], static_cast<size_t>(F) * N);
    if (rc == KWS_OK) rc = att_upload(&L.b_ff2, w->b_ff2[l], N);
    if (rc == KWS_OK) rc = att_upload(&L.ln2_g, w->ln2_g[l], N);
    if (rc == KWS_OK) rc = att_upload(&L.ln2_b, w->ln2_b[l], N);
    if (rc == KWS_OK && att_linear_tc_supported(N, 3 * N)) rc = att_pack_linear(w->w_qkv[l], N, 3 * N, &m->p_qkv[l].w, &m->p_qkv[l].nchunks);
    if (rc == KWS_OK && att_linear_tc_supported(N, F)) rc = att_pack_linear(w->w_ff1[l], N, F, &m->p_ff1[l].w, &m->p_ff1[l].nchunks);
    if (rc == KWS_OK && att_linear_tc_supported(F, N)) rc = att_pack_linear(w->w_ff2[l], F, N, &m->p_ff2[l].w, &m->p_ff2[l].nchunks);
  }
  if (rc == KWS_OK && att_linear_tc_supported(Kin, N)) rc = att_pack_linear(w->w_in, Kin, N, &m->p_in.w, &m->p_in.nchunks);
  if (rc == KWS_OK) rc = att_upload(&m->w_out, w->w_out, static_cast<size_t>(N) * C);
  if (rc == KWS_OK) rc = att_upload(&m->b_out, w->b_out, C);
  if (rc != KWS_OK) {
    att_free(m);
    return rc;
  }
  *out = m;
  return KWS_OK;
}

extern "C" int kws_attention_destroy(kws_attention* m) {
  clear_error();
  if (m) {
    cudaSetDevice(m->device);
    cudaDeviceSynchronize();
    att_free(m);
  }
  return KWS_OK;
}

extern "C" int32_t kws_attention_frames(const kws_attention* m, int32_t T) {
  return att_frames(T, m ? m->cfg.combine_frame : 2);   // models/attention_ctc.py:88-90
}

extern "C" int kws_attention_forward(kws_attention* m, const float* mel, int64_t B, int32_t T, float* probs_out,
                                     float* logits_out, void* stream) {
  return kws_attention_forward_lens(m, mel, B, T, nullptr, probs_out, logits_out, stream);
}

extern "C" int kws_attention_forward_lens(kws_attention* m, const float* mel, int64_t B, int32_t T, const int32_t* lens,
                                          float* probs_out, float* logits_out, void* stream) {
  clear_error();
  KWS_REQUIRE(m != nullptr, "model is NULL");
  KWS_REQUIRE(B >= 0 && T >= 1, "need at least one frame");
  if (B == 0) return KWS_OK;
  KWS_REQUIRE(mel && probs_out, "mel / probs_out is NULL");
  KWS_CUDA_OK(cudaSetDevice(m->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const auto& c = m->cfg;
  const int N = c.hidden, F = c.ffn, C = c.num_classes, Kin = c.n_mel * c.combine_frame;
  const int Tp = kws_attention_frames(m, T);
  const long rows = B * Tp;
  KWS_REQUIRE(rows < (1L << 31) / 4, "batch too large for one call (%ld rows): split it", rows);
  if (Tp > m->pe_rows) {                              // the K6 op: positional_encoding(max_length, hidden) (:96-97)
    KWS_CUDA_OK(cudaStreamSynchronize(st));
    cudaFree(m->pe);
    m->pe = nullptr;
    m->pe_rows = 0;
    KWS_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&m->pe), sizeof(float) * static_cast<size_t>(Tp) * N));
    m->pe_rows = Tp;
    const int rc = kws_positional_encoding(Tp, N, m->pe, stream);
    if (rc != KWS_OK) return rc;
  }
  // every segment starts on a 128-byte boundary: the tensor-core dense layers and the layer norm move 16-byte pieces,
  // and rows * Kin is odd for some accepted configs (n_mel = 41, combine_frame = 3 and an odd B * T')
  const auto seg = [rows](int width) { return (static_cast<size_t>(rows) * width + 31) & ~static_cast<size_t>(31); };
  const size_t scratch_floats = seg(Kin) + 3 * seg(N) + seg(F > 3 * N ? F : 3 * N);
  if (scratch_floats > m->scratch_floats) {
    KWS_CUDA_OK(cudaDeviceSynchronize());
    cudaFree(m->scratch);
    m->scratch = nullptr;
    m->scratch_floats = 0;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&m->scratch), sizeof(float) * scratch_floats);
    if (e != cudaSuccess) return fail(KWS_ERR_ALLOC, "scratch for %ld rows failed: %s", rows, cudaGetErrorString(e));
    m->scratch_floats = scratch_floats;
  }
  float* xin = m->scratch;
  float* x = xin + seg(Kin);
  float* y = x + seg(N);
  float* att = y + seg(N);
  float* big = att + seg(N);

  // layer norm: the utterance's T' * N floats in shared memory when they fit
  const size_t ln_bytes = sizeof(float) * static_cast<size_t>(Tp) * N;
  const int ln_in_smem = ln_bytes <= kLnSmemBytes ? 1 : 0;
  const size_t ln_smem = ln_in_smem ? ln_bytes : 0;
  KWS_CUDA_OK(cudaFuncSetAttribute(att_add_layernorm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLnSmemBytes));
  const AttLens L{lens, T, c.combine_frame};
  const long total_in = rows * Kin;
  att_combine_kernel<<<static_cast<unsigned>(ceil_div(total_in, 256)), 256, 0, st>>>(mel, B, T, c.n_mel, c.combine_frame, Tp,
                                                                                     L, xin);
  KWS_LAUNCH_OK("att_combine_kernel");
  int rc = att_linear<false, true>(xin, m->w_in, m->p_in, m->b_in, m->pe, Tp, L, rows, Kin, N, x, st);
  for (int l = 0; l < c.num_layers && rc == KWS_OK; ++l) {
    const auto& W = m->layer[l];
    rc = att_linear<false, false>(x, W.w_qkv, m->p_qkv[l], W.b_qkv, nullptr, Tp, L, rows, N, 3 * N, big, st);
    if (rc == KWS_OK) rc = att_core(big, B, Tp, c.heads, L, att, st);
    if (rc != KWS_OK) break;
    att_add_layernorm_kernel<<<static_cast<unsigned>(B), 1024, ln_smem, st>>>(att, x, W.ln1_g, W.ln1_b, Tp, L, N, ln_in_smem, y);
    KWS_LAUNCH_OK("att_add_layernorm_kernel");
    rc = att_linear<true, false>(y, W.w_ff1, m->p_ff1[l], W.b_ff1, nullptr, Tp, L, rows, N, F, big, st);
    if (rc == KWS_OK) rc = att_linear<false, false>(big, W.w_ff2, m->p_ff2[l], W.b_ff2, nullptr, Tp, L, rows, F, N, att, st);
    if (rc != KWS_OK) break;
    att_add_layernorm_kernel<<<static_cast<unsigned>(B), 1024, ln_smem, st>>>(att, y, W.ln2_g, W.ln2_b, Tp, L, N, ln_in_smem, x);
    KWS_LAUNCH_OK("att_add_layernorm_kernel");
  }
  if (rc != KWS_OK) return rc;
  att_output_kernel<<<static_cast<unsigned>(ceil_div(rows, 128)), 128, sizeof(float) * (N * C + C), st>>>(
      x, m->w_out, m->b_out, rows, Tp, L, N, C, c.use_relu, probs_out, logits_out);
  KWS_LAUNCH_OK("att_output_kernel");
  return KWS_OK;
}

// ---- single kernels of the forward pass on caller buffers, for tests that hold each one against a float64 reference
extern "C" int kws_debug_att_linear(const float* A, const float* W_host, const float* bias, const float* pe, int32_t Tp,
                                    int64_t rows, int32_t K, int32_t N, int relu, int add_pe, int path, float* Y,
                                    void* stream) {
  clear_error();
  KWS_REQUIRE(A && W_host && bias && Y && (pe || !add_pe), "NULL pointer");
  KWS_REQUIRE(rows >= 1 && K >= 1 && N >= 1 && Tp >= 1, "bad sizes");
  KWS_REQUIRE(path == 0 || path == 1, "path must be 0 (tcgen05) or 1 (FFMA)");
  if (path == 0 && !att_linear_tc_supported(K, N))
    return fail(KWS_ERR_UNSUPPORTED, "the tensor-core dense layer needs N %% 128 == 0 and K %% 4 == 0 (K = %d, N = %d)", K, N);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  kws_attention::Packed pk;
  float* dW = nullptr;
  int rc = path == 0 ? att_pack_linear(W_host, K, N, &pk.w, &pk.nchunks) : att_upload(&dW, W_host, static_cast<size_t>(K) * N);
  if (rc == KWS_OK) {
    const AttLens all{nullptr, Tp, 1};
    if (relu) rc = add_pe ? att_linear<true, true>(A, dW, pk, bias, pe, Tp, all, rows, K, N, Y, st)
                          : att_linear<true, false>(A, dW, pk, bias, pe, Tp, all, rows, K, N, Y, st);
    else rc = add_pe ? att_linear<false, true>(A, dW, pk, bias, pe, Tp, all, rows, K, N, Y, st)
                     : att_linear<false, false>(A, dW, pk, bias, pe, Tp, all, rows, K, N, Y, st);
  }
  const cudaError_t e = cudaStreamSynchronize(st);
  cudaFree(pk.w);
  cudaFree(dW);
  if (rc != KWS_OK) return rc;
  if (e != cudaSuccess) return fail(KWS_ERR_CUDA, "att_linear (path %d) failed: %s", path, cudaGetErrorString(e));
  return KWS_OK;
}

extern "C" int kws_debug_att_core(const float* qkv, int64_t B, int32_t Tp, int32_t heads, int path, float* out,
                                  void* stream) {
  return kws_debug_att_core_lens(qkv, B, Tp, nullptr, heads, path, out, stream);
}

extern "C" int kws_debug_att_core_lens(const float* qkv, int64_t B, int32_t Tp, const int32_t* lens, int32_t heads, int path,
                                       float* out, void* stream) {
  clear_error();
  KWS_REQUIRE(qkv && out, "NULL pointer");
  KWS_REQUIRE(B >= 1 && B <= 65535 && Tp >= 1 && heads >= 1 && heads <= 64, "bad sizes");
  KWS_REQUIRE(path == 0 || path == 1, "path must be 0 (tcgen05) or 1 (FFMA)");
  if (path == 0 && !att_core_tc_supported(Tp, heads, heads * kAttHeadDim))
    return fail(KWS_ERR_UNSUPPORTED, "the tensor-core attention core takes 1 <= T' <= 400 (T' = %d)", Tp);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const AttLens L{lens, Tp, 1};
  const int rc = path == 0 ? launch_att_core_tc(qkv, B, Tp, heads, L, out, st) : att_core_ffma(qkv, B, Tp, heads, L, 0, out, st);
  const cudaError_t e = cudaStreamSynchronize(st);
  if (rc != KWS_OK) return rc;
  if (e != cudaSuccess) return fail(KWS_ERR_CUDA, "attention core (path %d) failed: %s", path, cudaGetErrorString(e));
  return KWS_OK;
}

extern "C" int kws_debug_att_add_layernorm(const float* a, const float* b, const float* gamma, const float* beta,
                                           int64_t B, int32_t Tp, int32_t N, int in_smem, float* y, void* stream) {
  return kws_debug_att_add_layernorm_lens(a, b, gamma, beta, B, Tp, nullptr, N, in_smem, y, stream);
}

extern "C" int kws_debug_att_add_layernorm_lens(const float* a, const float* b, const float* gamma, const float* beta,
                                                int64_t B, int32_t Tp, const int32_t* lens, int32_t N, int in_smem, float* y,
                                                void* stream) {
  clear_error();
  KWS_REQUIRE(a && b && gamma && beta && y, "NULL pointer");
  KWS_REQUIRE(B >= 1 && B <= (1L << 31) - 1 && Tp >= 1 && N >= 1 && static_cast<int64_t>(Tp) * N < (1L << 31), "bad sizes");
  if (N % 4 != 0) return fail(KWS_ERR_UNSUPPORTED, "the layer norm needs N %% 4 == 0 (N = %d)", N);
  const size_t bytes = sizeof(float) * static_cast<size_t>(Tp) * N;
  if (in_smem && bytes > kLnSmemBytes)
    return fail(KWS_ERR_UNSUPPORTED, "T' * N = %d floats do not fit the layer norm's shared memory", Tp * N);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  KWS_CUDA_OK(cudaFuncSetAttribute(att_add_layernorm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLnSmemBytes));
  att_add_layernorm_kernel<<<static_cast<unsigned>(B), 1024, in_smem ? bytes : 0, st>>>(a, b, gamma, beta, Tp,
                                                                                       AttLens{lens, Tp, 1}, N, in_smem ? 1 : 0, y);
  KWS_LAUNCH_OK("att_add_layernorm_kernel");
  const cudaError_t e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return fail(KWS_ERR_CUDA, "att_add_layernorm_kernel failed: %s", cudaGetErrorString(e));
  return KWS_OK;
}
