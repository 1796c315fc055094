// K2+K3 -- persistent recurrent GRU (TF GRUCell semantics) + FC + softmax, fp32 path.
//
// Replaces inference1 / inference2 / tf.nn.softmax, models/rnn_ctc.py:156-165,202-284:
//   [r,u] = sigmoid([x,h] Wg + bg)          Wg [in+H, 2H]  (cols r | u)
//   c     = tanh([x, r*h] Wc + bc)          Wc [in+H, H]   (reset gate applied BEFORE the matmul)
//   h'    = u*h + (1-u)*c
//   last layer: softmax(h' Wfc + bfc)
// with dynamic_rnn(sequence_length) masking: past a stream's length the state is
// carried through and the output is zero (models/rnn_ctc.py:238-243).
//
// One CTA owns a tile of 64 streams for a whole layer and walks the time steps with
// h resident in registers + shared memory -- no HBM round trip of the state between
// steps.  The input projection x*W[0:in] is folded into the same K loop as the
// recurrent rows (rows of the TF kernels are already [x; h] ordered), so the
// [S*n, 384] pre-activations are never written to HBM.  Weights stream from L2 in
// 16-row blocks through a double-buffered shared-memory stage; thread (tx, ty) keeps
// an 8-stream x 4-unit register tile for r, u and c of the SAME hidden units, so the
// gate algebra needs no exchange.  This is the exact-fp32 (FFMA) path: it is the
// accuracy baseline for the tensor-core kernel and the always-available back end.
//
// launch_gru at the end is the host driver of all three back ends (this kernel, gru_tc.cu and gru_octbit.cu).
#include "common.cuh"

namespace kws {

constexpr int kTs = 64;        // streams per CTA tile
constexpr int kGruThreads = 256;
constexpr int kKb = 16;        // weight rows per staged block
constexpr int kH = kHidden;

struct GruLayerParams {
  int in_dim;
  long S;
  int n;                        // time steps
  // input: exactly one of x_rowmajor / x_tiled
  const float* x_rowmajor;      // [S, n, in_dim]
  const float* x_tiled;         // [tiles, n, in_dim(=H), 64]
  float* y_tiled;               // [tiles, n, H, 64] or null (last layer)
  float* y_rows;                // [S, n, H] row-major or null (the octbit graph's FC reads the last layer from here)
  const float* wg;              // [in+H, 2H]
  const float* bg;              // [2H]
  const float* wc;              // [in+H, H]
  const float* bc;              // [H]
  const float* h_in;            // [S, H]
  float* h_out;                 // [S, H]
  const int* seq_len;           // [S] or null
  const unsigned char* zero_state;  // [S] or null
  // last layer only
  const float* fc_w;            // [H, C]
  const float* fc_b;            // [C]
  int C;
  float* probs;                 // [S, n, C]
  float* logits;                // [S, n, C] or null
};

__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }

// acc[8][NC] += A[k][s0..s0+7] * W[k][cols], k over the virtual concat of two smem row blocks.
//   NC = 8: cols {4tx..4tx+3} and {H+4tx..H+4tx+3} of a 2H-wide W (gates);  NC = 4: cols 4tx..4tx+3 (candidate)
template <int NC>
__device__ __forceinline__ void tile_gemm(float (&acc)[8][NC], const float* __restrict__ A0, int n0,
                                          const float* __restrict__ A1, const float* __restrict__ W,
                                          int ktot, float* __restrict__ wb, int tx, int s0) {
  constexpr int LDW = NC == 8 ? 2 * kH : kH;
  constexpr int BLK4 = kKb * LDW / 4;                 // float4 per block
  constexpr int PF = BLK4 / kGruThreads;              // float4 per thread per block
  const int nblocks = (ktot + kKb - 1) / kKb;
  const long wlimit4 = static_cast<long>(ktot) * LDW / 4;
  const float4* W4 = reinterpret_cast<const float4*>(W);
  float4 pf[PF];
  // block 0 -> buffer 0
#pragma unroll
  for (int q = 0; q < PF; ++q) {
    const long i = threadIdx.x + q * kGruThreads;
    pf[q] = i < wlimit4 ? __ldg(W4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    reinterpret_cast<float4*>(wb)[threadIdx.x + q * kGruThreads] = pf[q];
  }
  __syncthreads();
  for (int b = 0; b < nblocks; ++b) {
    const bool more = b + 1 < nblocks;
    if (more) {
#pragma unroll
      for (int q = 0; q < PF; ++q) {
        const long i = static_cast<long>(b + 1) * BLK4 + threadIdx.x + q * kGruThreads;
        pf[q] = i < wlimit4 ? __ldg(W4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    const float* wcur = wb + (b & 1) * (kKb * LDW);
    const int rows = min(kKb, ktot - b * kKb);
#pragma unroll
    for (int kk = 0; kk < kKb; ++kk) {
      if (kk < rows) {
        const int k = b * kKb + kk;
        const float* arow = (k < n0 ? A0 + k * kTs : A1 + (k - n0) * kTs) + s0;
        const float4 a0 = *reinterpret_cast<const float4*>(arow);
        const float4 a1 = *reinterpret_cast<const float4*>(arow + 4);
        const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        const float4 w0 = *reinterpret_cast<const float4*>(wcur + kk * LDW + 4 * tx);
        float w[NC];
        w[0] = w0.x; w[1] = w0.y; w[2] = w0.z; w[3] = w0.w;
        if (NC == 8) {
          const float4 w1 = *reinterpret_cast<const float4*>(wcur + kk * LDW + kH + 4 * tx);
          w[NC - 4] = w1.x; w[NC - 3] = w1.y; w[NC - 2] = w1.z; w[NC - 1] = w1.w;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int c = 0; c < NC; ++c) acc[i][c] = fmaf(a[i], w[c], acc[i][c]);
      }
    }
    if (more) {
      float4* wnext = reinterpret_cast<float4*>(wb + ((b + 1) & 1) * (kKb * LDW));
#pragma unroll
      for (int q = 0; q < PF; ++q) wnext[threadIdx.x + q * kGruThreads] = pf[q];
    }
    __syncthreads();
  }
}

template <bool kLast>
__global__ void __launch_bounds__(kGruThreads, 1)
gru_layer_kernel(const GruLayerParams p) {
  extern __shared__ __align__(16) float smem[];
  float* Xs = smem;                               // [in_dim][64]
  float* Hs = Xs + p.in_dim * kTs;                // [H][64]
  float* RHs = Hs + kH * kTs;                     // [H][64]
  float* Wb = RHs + kH * kTs;                     // [2][16*2H]
  float* fcw = Wb + 2 * kKb * 2 * kH;             // [H*C]      (last layer)
  float* fcb = fcw + kH * kMaxClasses;            // [16]
  float* Lg = fcb + kMaxClasses;                  // [64][C]

  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int s0 = ty * 8, j0 = tx * 4;
  const int ktot = p.in_dim + kH;
  const long ntiles = (p.S + kTs - 1) / kTs;

  float bgr[4], bgu[4], bcc[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    bgr[c] = p.bg[j0 + c];
    bgu[c] = p.bg[kH + j0 + c];
    bcc[c] = p.bc[j0 + c];
  }
  if (kLast) {
    for (int i = threadIdx.x; i < kH * p.C; i += kGruThreads) fcw[i] = p.fc_w[i];
    if (threadIdx.x < p.C) fcb[threadIdx.x] = p.fc_b[threadIdx.x];
  }

  for (long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long sbase = tile * kTs;
    // ---- carried state -> registers + smem
    float h[8][4];
    int len[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const long s = sbase + s0 + i;
      const bool ok = s < p.S;
      const bool zero = ok && p.zero_state && p.zero_state[s];
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ok && !zero) v = *reinterpret_cast<const float4*>(p.h_in + s * kH + j0);
      h[i][0] = v.x; h[i][1] = v.y; h[i][2] = v.z; h[i][3] = v.w;
      len[i] = ok ? (p.seq_len ? p.seq_len[s] : p.n) : 0;
    }
    __syncthreads();   // previous tile's readers of Hs are done
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      *reinterpret_cast<float4*>(Hs + (j0 + c) * kTs + s0) = make_float4(h[0][c], h[1][c], h[2][c], h[3][c]);
      *reinterpret_cast<float4*>(Hs + (j0 + c) * kTs + s0 + 4) = make_float4(h[4][c], h[5][c], h[6][c], h[7][c]);
    }

    for (int t = 0; t < p.n; ++t) {
      // ---- x_t -> Xs[k][s]
      if (p.x_tiled) {
        const float4* src = reinterpret_cast<const float4*>(p.x_tiled + (tile * p.n + t) * static_cast<long>(p.in_dim) * kTs);
        float4* dst = reinterpret_cast<float4*>(Xs);
        for (int i = threadIdx.x; i < p.in_dim * kTs / 4; i += kGruThreads) dst[i] = __ldg(src + i);
      } else {
        const int sl = threadIdx.x & 63, part = threadIdx.x >> 6;
        const long s = sbase + sl;
        const bool ok = s < p.S;
        const float* row = p.x_rowmajor + (ok ? (s * p.n + t) * static_cast<long>(p.in_dim) : 0);
        if ((p.in_dim & 3) == 0) {
          for (int q = part; q < p.in_dim / 4; q += 4) {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (ok) v = __ldg(reinterpret_cast<const float4*>(row) + q);
            Xs[(4 * q + 0) * kTs + sl] = v.x;
            Xs[(4 * q + 1) * kTs + sl] = v.y;
            Xs[(4 * q + 2) * kTs + sl] = v.z;
            Xs[(4 * q + 3) * kTs + sl] = v.w;
          }
        } else {
          for (int k = part; k < p.in_dim; k += 4) Xs[k * kTs + sl] = ok ? __ldg(row + k) : 0.0f;
        }
      }
      __syncthreads();

      // ---- gates
      float g[8][8];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int c = 0; c < 8; ++c) g[i][c] = 0.0f;
      tile_gemm<8>(g, Xs, p.in_dim, Hs, p.wg, ktot, Wb, tx, s0);
      float u[8][4];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float r = sigmoid_f(g[i][c] + bgr[c]);
          u[i][c] = sigmoid_f(g[i][4 + c] + bgu[c]);
          g[i][c] = r * h[i][c];                       // r (.) h, input of the candidate matmul
        }
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        *reinterpret_cast<float4*>(RHs + (j0 + c) * kTs + s0) = make_float4(g[0][c], g[1][c], g[2][c], g[3][c]);
        *reinterpret_cast<float4*>(RHs + (j0 + c) * kTs + s0 + 4) = make_float4(g[4][c], g[5][c], g[6][c], g[7][c]);
      }
      __syncthreads();

      // ---- candidate + state update
      float cc[8][4];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int c = 0; c < 4; ++c) cc[i][c] = 0.0f;
      tile_gemm<4>(cc, Xs, p.in_dim, RHs, p.wc, ktot, Wb, tx, s0);
      float y[8][4];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const bool live = t < len[i];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float cand = tanhf(cc[i][c] + bcc[c]);
          const float hn = u[i][c] * h[i][c] + (1.0f - u[i][c]) * cand;
          h[i][c] = live ? hn : h[i][c];
          y[i][c] = live ? hn : 0.0f;
        }
      }
      // h for the next step's gate matmul
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        *reinterpret_cast<float4*>(Hs + (j0 + c) * kTs + s0) = make_float4(h[0][c], h[1][c], h[2][c], h[3][c]);
        *reinterpret_cast<float4*>(Hs + (j0 + c) * kTs + s0 + 4) = make_float4(h[4][c], h[5][c], h[6][c], h[7][c]);
      }
      if (!kLast) {
        if (p.y_tiled) {
          float* dst = p.y_tiled + ((tile * p.n + t) * static_cast<long>(kH)) * kTs;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            *reinterpret_cast<float4*>(dst + (j0 + c) * kTs + s0) = make_float4(y[0][c], y[1][c], y[2][c], y[3][c]);
            *reinterpret_cast<float4*>(dst + (j0 + c) * kTs + s0 + 4) = make_float4(y[4][c], y[5][c], y[6][c], y[7][c]);
          }
        }
        if (p.y_rows) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const long s = sbase + s0 + i;
            if (s < p.S)
              *reinterpret_cast<float4*>(p.y_rows + (s * p.n + t) * kH + j0) = make_float4(y[i][0], y[i][1], y[i][2], y[i][3]);
          }
        }
      } else {
        // outputs (zero past seq_len) -> RHs as the FC input; RHs is free until the next step's gates
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          *reinterpret_cast<float4*>(RHs + (j0 + c) * kTs + s0) = make_float4(y[0][c], y[1][c], y[2][c], y[3][c]);
          *reinterpret_cast<float4*>(RHs + (j0 + c) * kTs + s0 + 4) = make_float4(y[4][c], y[5][c], y[6][c], y[7][c]);
        }
      }
      __syncthreads();

      if (kLast) {
        // ---- FC: logits[s][c] = sum_j y[j][s] * fcw[j][c] + b[c]
        const int sl = threadIdx.x & 63, cq = threadIdx.x >> 6;
        for (int c = cq; c < p.C; c += 4) {
          float acc = 0.0f;
#pragma unroll 8
          for (int j = 0; j < kH; ++j) acc = fmaf(RHs[j * kTs + sl], fcw[j * p.C + c], acc);
          Lg[sl * p.C + c] = acc + fcb[c];
        }
        __syncthreads();
        if (threadIdx.x < kTs) {
          const long s = sbase + threadIdx.x;
          if (s < p.S) {
            float lg[kMaxClasses];
            float mx = -INFINITY;
            for (int c = 0; c < p.C; ++c) {
              lg[c] = Lg[threadIdx.x * p.C + c];
              mx = fmaxf(mx, lg[c]);
            }
            float sum = 0.0f;
            float e[kMaxClasses];
            for (int c = 0; c < p.C; ++c) {
              e[c] = expf(lg[c] - mx);
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
        // Lg is rewritten only after the next step's barriers; no extra sync needed here
      }
    }
    // ---- final state
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const long s = sbase + s0 + i;
      if (s < p.S)
        *reinterpret_cast<float4*>(p.h_out + s * kH + j0) = make_float4(h[i][0], h[i][1], h[i][2], h[i][3]);
    }
  }
}

static size_t gru_smem_bytes(int in_dim) {
  return sizeof(float) * (static_cast<size_t>(in_dim) * kTs + 2 * kH * kTs + 2 * kKb * 2 * kH +
                          kH * kMaxClasses + kMaxClasses + kTs * kMaxClasses);
}

// One layer of the fp32 path.  x_tiled: the layer below in the tiled hand-off layout (null for layer 0, which reads
// a.x row-major); y_tiled / y_rows: where the layer's outputs go when it does not run the FC itself (either may be
// null); fused_fc: the last layer of the float graph, FC + softmax in the same kernel.
static int launch_layer_fp32(kws_model* m, const GruArgs& a, int l, const float* x_tiled, float* y_tiled, float* y_rows,
                             bool fused_fc, cudaStream_t st) {
  const long ntiles = ceil_div(a.S, kTs);
  GruLayerParams p;
  p.in_dim = m->layer[l].in_dim;
  p.S = a.S;
  p.n = a.n;
  p.x_rowmajor = l == 0 ? a.x : nullptr;
  p.x_tiled = l == 0 ? nullptr : x_tiled;
  p.y_tiled = y_tiled;
  p.y_rows = y_rows;
  p.wg = m->layer[l].gates_kernel;
  p.bg = m->layer[l].gates_bias;
  p.wc = m->layer[l].cand_kernel;
  p.bc = m->layer[l].cand_bias;
  p.h_in = a.state_in + static_cast<long>(l) * a.S * kH;
  p.h_out = a.state_out + static_cast<long>(l) * a.S * kH;
  p.seq_len = a.seq_len;
  p.zero_state = a.zero_state;
  p.fc_w = m->fc_w;
  p.fc_b = m->fc_b;
  p.C = m->cfg.num_classes;
  p.probs = a.probs;
  p.logits = a.logits;
  const size_t smem = gru_smem_bytes(p.in_dim);
  long blocks = ntiles < sm_count() ? ntiles : sm_count();
  if (fused_fc) {
    KWS_CUDA_OK(cudaFuncSetAttribute(gru_layer_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     static_cast<int>(smem)));
    gru_layer_kernel<true><<<static_cast<unsigned>(blocks), kGruThreads, smem, st>>>(p);
  } else {
    KWS_CUDA_OK(cudaFuncSetAttribute(gru_layer_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     static_cast<int>(smem)));
    gru_layer_kernel<false><<<static_cast<unsigned>(blocks), kGruThreads, smem, st>>>(p);
  }
  KWS_LAUNCH_OK("gru_layer_kernel");
  return KWS_OK;
}

// zero the carried state of the streams flagged by zero_state (a call without frames)
__global__ void zero_flagged_state_kernel(float* state, long S, int layers, const unsigned char* flags) {
  const long idx = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  const long total = static_cast<long>(layers) * S * kH;
  if (idx >= total) return;
  const long s = (idx / kH) % S;
  if (flags[s]) state[idx] = 0.0f;
}

int launch_gru(kws_model* m, const GruArgs& a, cudaStream_t st) {
  if (a.S <= 0) return KWS_OK;
  const int L = m->cfg.num_layers;
  if (a.n <= 0) {
    if (a.state_out != a.state_in)
      KWS_CUDA_OK(cudaMemcpyAsync(a.state_out, a.state_in, sizeof(float) * L * a.S * kH, cudaMemcpyDeviceToDevice, st));
    if (a.zero_state) {
      const long total = static_cast<long>(L) * a.S * kH;
      zero_flagged_state_kernel<<<static_cast<unsigned>(ceil_div(total, 256)), 256, 0, st>>>(a.state_out, a.S, L,
                                                                                              a.zero_state);
      KWS_LAUNCH_OK("zero_flagged_state_kernel");
    }
    return KWS_OK;
  }
  if (L > 1 && !a.seq_scratch) {
    const int rc = kws_model_reserve(m, a.S, a.n);
    if (rc != KWS_OK) return rc;
  }
  float* seq = a.seq_scratch ? a.seq_scratch : m->scratch_seq;
  if (model_uses_tc(m)) return launch_gru_tc(m, a, seq, st);

  // CUDA cores.  The float graph fuses the FC into its last layer; the octbit graph's last layer writes y_rows for
  // fc_octbit_softmax_kernel.  Layers the rewriter left in fp32 (cell_0) run the fp32 kernel in either graph.
  float* y_rows = nullptr;
  if (m->octbit) {
    y_rows = a.y_rows_scratch;
    if (!y_rows) {
      const int rc = grow_scratch(reinterpret_cast<void**>(&m->oct_y_rows), &m->oct_y_bytes,
                                  sizeof(float) * a.S * a.n * kH, "octbit FC input scratch");
      if (rc != KWS_OK) return rc;
      y_rows = m->oct_y_rows;
    }
  }
  const long per_buf = ceil_div(a.S, kTs) * a.n * static_cast<long>(kH) * kTs;
  for (int l = 0; l < L; ++l) {
    const bool last = l == L - 1;
    const float* x_tiled = l == 0 ? nullptr : seq + ((l - 1) & 1) * per_buf;
    float* y_tiled = last ? nullptr : seq + (l & 1) * per_buf;
    float* yr = last ? y_rows : nullptr;
    const int rc = m->oct_gates[l].wq ? launch_octbit_layer(m, a, l, x_tiled, y_tiled, yr, st)
                                      : launch_layer_fp32(m, a, l, x_tiled, y_tiled, yr, last && !m->octbit, st);
    if (rc != KWS_OK) return rc;
  }
  return m->octbit ? launch_octbit_fc(m, a, y_rows, st) : KWS_OK;
}

}  // namespace kws
