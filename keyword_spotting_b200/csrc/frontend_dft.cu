// K1 for every frame other than 400/160: framing + |real DFT_N| + mel as one tcgen05 GEMM per 128 frames, with the
// magnitude and the mel projection on the CUDA cores.
//
// Replaces the same reference lines as frontend.cu (utils/stft.py:27-81, models/rnn_ctc.py:135-149) for a frame of
// N = fft_size samples (16 <= N <= 512) at any hop_size in [1, N].  The real DFT of N samples has exactly N real
// outputs (cos bins 0 .. floor(N/2), sin bins 1 .. ceil(N/2) - 1), so the spectra of 128 frames are one product
//     D[frame, col] = sum_m x_frame[m] W[col, m]        (tcgen05.mma kind::f16, M = 128 frames, N = ncols, K = N)
// with a constant twiddle matrix W.  Columns: cos bin k at column k (k < Hc = ceil(N/2)), sin bin k at column
// B + k (0 < k < Hc, B = ceil16(Hc)), and for even N the Nyquist cos bin at column B (where sin 0 = 0 would be).
// ncols = ceil16(B + Hc) <= 512 fp32 accumulator columns: one TMEM allocation of 512 columns at N <= 512.
//
//   rows   (stream, frame) pairs flattened over the batch: row r of mel_out [S, max_frames, n_mel] is tile r / 128,
//          lane r % 128, so one tile spans several streams when a stream has few frames (a streaming chunk).
//   K      in chunks of 32 samples, two stages: the PCM rows are staged by the 128 threads (thread = row, element by
//          element, since frames overlap and hop need not be a multiple of 8) while the previous chunk's MMAs run; the
//          twiddle chunk (pre-packed at model creation, hi and lo, ncols x 32 each) arrives by one bulk copy.  At
//          N = 512 the whole matrix is 1 MB, so it is streamed per chunk and read from L2.
//   exact  int16 x = x_hi + x_lo exactly in fp16 (x_hi = fp16(x), |x_lo| <= 16); fp32 PCM is scaled by 2^15 first
//          (exact) and split to 2^-22 of |x| -- so |x| must stay below 2 (fp16 range).  W = W_hi + W_lo; three MMAs
//          per K step (x_hi W_hi + x_lo W_hi + x_hi W_lo), accumulated in fp32: the accuracy of an fp32 transform.
//   epilogue  thread = row: |X_k| = sqrt(c^2 + s^2) from TMEM into a [128][bins] shared array (over the stage
//          buffers), then mel[band] = sum_k basis[k, band] |X_k| over the band's non-zero span with warp-broadcast
//          weights, x 2^-15, into a [128][n_mel] tile that leaves through FrontendIo::store_tile / zero_rows.
//   dead tiles  a tile with no row below its stream's frame count (under lengths) loads no PCM and issues no MMA.
//
// The streaming server's VAD / next-tail pre-step is not fused here (frontend_can_fuse_pre is false for these models):
// stream_pre_kernel runs it before this kernel.
#include <cmath>
#include <vector>

#include <cuda_fp16.h>

#include "frontend_io.cuh"

namespace kws {

constexpr int kDfThreads = 128;               // thread = tile row = TMEM lane
constexpr int kDfKc = 32;                     // samples per K chunk
constexpr int kDfSbo = (kDfKc / 8) * 128;     // 512 bytes between 8-row groups of an operand chunk
constexpr int kDfAPart = kDfThreads * kDfKc * 2;   // 8 KB: one fp16 part of the PCM operand chunk

struct FrontendDftParams : FrontendIo {
  const uint4* tw;          // [chunks][hi | lo][ncols x 32 canonical K-major] fp16
  const int4* mel_seg;      // [n_mel] {first bin, bins, offset into mel_w, 0}
  const float* mel_w;       // the bands' non-zero spans, concatenated
  int fft, hop;
  int chunks;               // ceil(fft / 32)
  int ncols;                // accumulator columns (multiple of 16, <= 512)
  int hc, bcol;             // Hc = ceil(N/2), B = ceil16(Hc)
  int ldm, ldo;             // floats per row of the magnitude array (odd) and of the output tile (odd)
  uint32_t tmem_cols;
  long rows;                // S * max_frames
};

__device__ __forceinline__ int df_frames(const FrontendDftParams& p, int total) {
  const int n = frames_of(total, p.fft, p.hop);
  return n < p.max_frames ? n : p.max_frames;
}

template <bool kLens, bool kI16>
__global__ void __launch_bounds__(kDfThreads, 1)
frontend_dft_kernel(const FrontendDftParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int stage_bytes = 2 * kDfAPart + p.ncols * 128;
  const int region_bytes = max(2 * stage_bytes, kDfThreads * p.ldm * 4);
  float* sMag = reinterpret_cast<float*>(smem);                          // over the stage buffers
  float* sOut = reinterpret_cast<float*>(smem + region_bytes);           // [128][ldo]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sOut + kDfThreads * p.ldo);   // tw_full[2], mma_done[2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);

  const int tid = threadIdx.x, warp = tid >> 5;
  if (warp == 0) tc::tmem_alloc(tmem_slot, p.tmem_cols);
  if (tid == 0) {
    for (int i = 0; i < 4; ++i) tc::mbar_init(&bars[i], 1);
    tc::mbar_fence_init();
  }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const uint32_t lane_sel = static_cast<uint32_t>(32 * warp) << 16;

  const int N = p.fft, M = p.n_mel, mf = p.max_frames;
  const uint32_t chunk_bytes = static_cast<uint32_t>(p.ncols) * 128;
  const int pieces = (p.ncols + 255) / 256;
  const long tiles = (p.rows + kDfThreads - 1) / kDfThreads;
  uint32_t g = 0;                                  // K chunks issued by this CTA: stage g & 1, barrier phase g >> 1

  for (long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const long r0 = tile * kDfThreads;
    const long r = r0 + tid;
    // this row's stream, frame and whether the frame exists
    long s = 0;
    int f = 0, head_len = 0, nfr = 0;
    if (r < p.rows) {
      s = r / mf;
      f = static_cast<int>(r - s * mf);
      head_len = p.src.head_len ? __ldg(p.src.head_len + s) : 0;
      nfr = df_frames(p, p.total_len<kLens>(s, head_len));
      if (kLens && p.nframes_out && f == 0) p.nframes_out[s] = nfr;
    }
    const bool live = f < nfr;
    const bool tile_live = __syncthreads_or(live) != 0;

    if (tile_live) {
      const int16_t* head = p.src.head ? p.src.head + s * p.src.ld_head : nullptr;
      const long pos0 = static_cast<long>(f) * p.hop;           // the frame's first sample in the stream
      for (int c = 0; c < p.chunks; ++c, ++g) {
        const int buf = static_cast<int>(g & 1);
        unsigned char* stage = smem + buf * stage_bytes;
        if (g >= 2) tc::mbar_wait(&bars[2 + buf], ((g >> 1) - 1) & 1);   // the MMAs that read this stage are done
        if (warp == 0) {
          if (tc::elect_one()) {
            tc::mbar_arrive_expect_tx(&bars[buf], chunk_bytes);
            tc::bulk_g2s(stage + 2 * kDfAPart, p.tw + static_cast<long>(c) * (chunk_bytes / 16), chunk_bytes, &bars[buf]);
          }
          __syncwarp();
        }
        // this row's 32 samples of the chunk -> fp16 hi / lo, four 16-byte core-matrix rows per part
        const int k0 = c * kDfKc;
#pragma unroll
        for (int q = 0; q < kDfKc / 8; ++q) {
          float v[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int k = k0 + 8 * q + j;
            float x = 0.0f;
            if (live && k < N) {
              const long pos = pos0 + k;                        // < the stream's length: the frame exists
              if (pos < head_len) {
                x = static_cast<float>(head[pos]);
              } else if (kI16) {
                x = static_cast<float>(__ldg(static_cast<const int16_t*>(p.src.body) + s * p.src.ld_body + (pos - head_len)));
              } else {
                x = __ldg(static_cast<const float*>(p.src.body) + s * p.src.ld_body + (pos - head_len)) * 32768.0f;
              }
            }
            v[j] = x;
          }
          uint4 hi, lo;
          tc::split_half8(v, &hi, &lo);
          const int off = (tid >> 3) * kDfSbo + q * 128 + (tid & 7) * 16;
          *reinterpret_cast<uint4*>(stage + off) = hi;
          *reinterpret_cast<uint4*>(stage + kDfAPart + off) = lo;
        }
        tc::fence_proxy_async();
        __syncthreads();
        if (warp == 0) {
          tc::mbar_wait(&bars[buf], (g >> 1) & 1);
          tc::fence_after_sync();
          if (tc::elect_one()) {
            const uint32_t base = tc::smem_u32(stage);
            const uint64_t a_hi = tc::smem_desc(base, 128, kDfSbo), a_lo = a_hi + (kDfAPart >> 4);
            const uint64_t b_hi = tc::smem_desc(base + 2 * kDfAPart, 128, kDfSbo), b_lo = b_hi + ((chunk_bytes / 2) >> 4);
#pragma unroll
            for (int ks = 0; ks < kDfKc / 16; ++ks) {
              const uint64_t step = static_cast<uint64_t>(ks * (256 >> 4));
              for (int pc = 0; pc < pieces; ++pc) {
                const int n = min(256, p.ncols - 256 * pc);
                const uint32_t idesc = tc::idesc_f16(128, n);
                const uint32_t d = tmem + 256 * pc;
                const uint64_t bo = step + static_cast<uint64_t>(pc * ((32 * kDfSbo) >> 4));   // rows 256 pc ..
                tc::mma_ss(d, a_hi + step, b_hi + bo, idesc, c > 0 || ks > 0);
                tc::mma_ss(d, a_lo + step, b_hi + bo, idesc, true);
                tc::mma_ss(d, a_hi + step, b_lo + bo, idesc, true);
              }
            }
            tc::commit(&bars[2 + buf]);
          }
          __syncwarp();
        }
      }
      // ---- magnitudes: thread = row, straight from TMEM
      tc::mbar_wait(&bars[2 + ((g - 1) & 1)], ((g - 1) >> 1) & 1);
      tc::fence_after_sync();
      float* mrow = sMag + tid * p.ldm;
      for (int j0 = 0; j0 < p.hc; j0 += 16) {
        uint32_t cv[16], sv[16];
        tc::ld16(tmem + lane_sel + j0, cv);
        tc::ld16(tmem + lane_sel + p.bcol + j0, sv);
        tc::wait_ld();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int k = j0 + j;
          const float cr = __uint_as_float(cv[j]), si = k == 0 ? 0.0f : __uint_as_float(sv[j]);
          if (k < p.hc) mrow[k] = sqrtf(fmaf(cr, cr, si * si));
        }
        if (j0 == 0 && (N & 1) == 0) mrow[p.hc] = fabsf(__uint_as_float(sv[0]));   // Nyquist bin N/2
      }
      tc::fence_before_sync();
      // ---- mel projection of this row (its own magnitudes: no barrier between the two)
      float* orow = sOut + tid * p.ldo;
#pragma unroll 1
      for (int band = 0; band < M; ++band) {
        const int4 seg = __ldg(p.mel_seg + band);
        const float* w = p.mel_w + seg.z;
        const float* mg = mrow + seg.x;
        float a0 = 0.0f, a1 = 0.0f;
        int j = 0;
#pragma unroll 1
        for (; j + 1 < seg.y; j += 2) {
          a0 = fmaf(__ldg(w + j), mg[j], a0);
          a1 = fmaf(__ldg(w + j + 1), mg[j + 1], a1);
        }
        if (j < seg.y) a0 = fmaf(__ldg(w + j), mg[j], a0);
        orow[band] = (a0 + a1) * 3.0517578125e-05f;                  // 2^-15 (detector.py:40-43)
      }
      tc::fence_proxy_async();                                       // the next chunk's bulk copy lands over sMag
    }
    __syncthreads();
    // ---- the tile's rows, stream by stream
    const long rend = r0 + kDfThreads < p.rows ? r0 + kDfThreads : p.rows;
    for (long ss = r0 / mf; ss * mf < rend; ++ss) {
      const int fa = static_cast<int>(max(r0 - ss * mf, 0L));
      const int fb = static_cast<int>(min(rend - ss * mf, static_cast<long>(mf)));
      const int hl = p.src.head_len ? __ldg(p.src.head_len + ss) : 0;
      const int n_s = df_frames(p, p.total_len<kLens>(ss, hl));
      const int nst = min(fb, n_s);
      if (tile_live && nst > fa)
        p.store_tile<kDfThreads>(sOut + (ss * mf + fa - r0) * p.ldo, p.ldo, ss, fa, nst - fa, tid);
      if (kLens) p.zero_rows<kDfThreads>(ss, max(fa, n_s), fb, tid);   // rows past the stream's length
    }
    __syncthreads();
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem, p.tmem_cols);
}

namespace {
struct DftGeom {
  int hc, bcol, ncols, chunks;
};
DftGeom dft_geom(int N) {
  DftGeom d;
  d.hc = (N + 1) / 2;
  d.bcol = (d.hc + 15) / 16 * 16;
  d.ncols = (d.bcol + d.hc + 15) / 16 * 16;
  d.chunks = (N + kDfKc - 1) / kDfKc;
  return d;
}
}  // namespace

// Twiddles of an N-point real DFT as the B operand of every K chunk ([ncols, 32] K-major canonical, fp16 hi then lo),
// and the non-zero span of every mel band of a basis [N/2 + 1, M].
int build_frontend_dft_tables(kws_model* m, const float* basis) {
  const int N = m->cfg.fft_size, M = m->cfg.n_mel, nb = N / 2 + 1;
  const DftGeom d = dft_geom(N);
  const size_t part = static_cast<size_t>(d.ncols) * kDfKc;        // halves per part of one chunk
  std::vector<__half> tw(static_cast<size_t>(d.chunks) * 2 * part, __float2half_rn(0.0f));
  for (int col = 0; col < d.ncols; ++col) {
    for (int mm = 0; mm < N; ++mm) {
      double v = 0.0;
      if (col < d.hc) {
        v = std::cos(2.0 * M_PI * static_cast<double>((static_cast<long>(mm) * col) % N) / N);
      } else if (col == d.bcol) {
        v = (N & 1) == 0 ? ((mm & 1) ? -1.0 : 1.0) : 0.0;            // cos(pi m): the Nyquist bin of an even N
      } else if (col > d.bcol && col < d.bcol + d.hc) {
        v = -std::sin(2.0 * M_PI * static_cast<double>((static_cast<long>(mm) * (col - d.bcol)) % N) / N);
      }
      const __half hi = __float2half_rn(static_cast<float>(v));
      const __half lo = __float2half_rn(static_cast<float>(v - static_cast<double>(__half2float(hi))));
      const size_t base = static_cast<size_t>(mm / kDfKc) * 2 * part;
      const size_t off = tc::canon_offset(col, mm % kDfKc, kDfKc) / 2;
      tw[base + off] = hi;
      tw[base + part + off] = lo;
    }
  }
  std::vector<int4> seg(M);
  std::vector<float> wts;
  for (int band = 0; band < M; ++band) {
    int lo = -1, hi = -1;
    for (int k = 0; k < nb; ++k)
      if (basis[static_cast<size_t>(k) * M + band] != 0.0f) {
        if (lo < 0) lo = k;
        hi = k;
      }
    const int n = lo < 0 ? 0 : hi - lo + 1;                  // an all-zero band sums nothing
    seg[band] = make_int4(lo < 0 ? 0 : lo, n, static_cast<int>(wts.size()), 0);
    for (int j = 0; j < n; ++j) wts.push_back(basis[static_cast<size_t>(lo + j) * M + band]);
  }
  if (wts.empty()) wts.push_back(0.0f);
  KWS_CUDA_OK(cudaMalloc(&m->fe_dft.tw, tw.size() * sizeof(__half)));
  KWS_CUDA_OK(cudaMemcpy(m->fe_dft.tw, tw.data(), tw.size() * sizeof(__half), cudaMemcpyHostToDevice));
  KWS_CUDA_OK(cudaMalloc(&m->fe_dft.mel_seg, seg.size() * sizeof(int4)));
  KWS_CUDA_OK(cudaMemcpy(m->fe_dft.mel_seg, seg.data(), seg.size() * sizeof(int4), cudaMemcpyHostToDevice));
  KWS_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&m->fe_dft.mel_w), wts.size() * sizeof(float)));
  KWS_CUDA_OK(cudaMemcpy(m->fe_dft.mel_w, wts.data(), wts.size() * sizeof(float), cudaMemcpyHostToDevice));
  return KWS_OK;
}

void free_frontend_dft_tables(kws_model* m) {
  cudaFree(m->fe_dft.tw);
  cudaFree(m->fe_dft.mel_seg);
  cudaFree(m->fe_dft.mel_w);
  m->fe_dft = FrontendDftTables();
}

int launch_frontend_dft(const kws_model* m, const FrontendIo& io, cudaStream_t st) {
  if (io.fuse_pre) return fail(KWS_ERR_INVALID_ARGUMENT, "the DFT front end takes no fused pre-step");
  FrontendDftParams p{io};
  const int N = m->cfg.fft_size, M = m->cfg.n_mel;
  const DftGeom d = dft_geom(N);
  p.tw = static_cast<const uint4*>(m->fe_dft.tw);
  p.mel_seg = static_cast<const int4*>(m->fe_dft.mel_seg);
  p.mel_w = m->fe_dft.mel_w;
  p.fft = N;
  p.hop = m->cfg.hop_size;
  p.chunks = d.chunks;
  p.ncols = d.ncols;
  p.hc = d.hc;
  p.bcol = d.bcol;
  p.ldm = (N / 2 + 1) | 1;
  p.ldo = M | 1;
  uint32_t cols = 32;
  while (static_cast<int>(cols) < 2 * d.bcol) cols *= 2;           // every column the epilogue reads
  p.tmem_cols = cols;
  p.rows = io.S * static_cast<long>(io.max_frames);
  if (p.rows <= 0) return KWS_OK;
  const int stage_bytes = 2 * kDfAPart + d.ncols * 128;
  const size_t region = std::max(2 * stage_bytes, kDfThreads * p.ldm * 4);
  const size_t smem = region + sizeof(float) * kDfThreads * p.ldo + 4 * sizeof(uint64_t) + 16;
  const bool i16 = io.src.body_dtype == KWS_PCM_I16, lens = io.src.lengths != nullptr;
  auto kernel = lens ? (i16 ? frontend_dft_kernel<true, true> : frontend_dft_kernel<true, false>)
                     : (i16 ? frontend_dft_kernel<false, true> : frontend_dft_kernel<false, false>);
  KWS_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  int per_sm = 0;
  KWS_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kDfThreads, smem));
  if (per_sm < 1) return fail(KWS_ERR_CUDA, "frontend_dft_kernel does not fit on an SM (smem %zu)", smem);
  if (per_sm > static_cast<int>(512 / cols)) per_sm = static_cast<int>(512 / cols);   // TMEM: 512 columns per SM
  const long tiles = (p.rows + kDfThreads - 1) / kDfThreads;
  long blocks = static_cast<long>(per_sm) * sm_count();
  if (blocks > tiles) blocks = tiles;
  kernel<<<static_cast<unsigned>(blocks), kDfThreads, smem, st>>>(p);
  KWS_LAUNCH_OK("frontend_dft_kernel");
  return KWS_OK;
}

}  // namespace kws
