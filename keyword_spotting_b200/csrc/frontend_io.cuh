// What the two front-end kernels (frontend.cu: FFT, frontend_tc.cu: tensor cores) share around their transforms: the
// launch parameters, a stream's length and frame count, the copy of a finished [frames, n_mel] tile into mel_out in
// its three layouts, the zero rows past a stream's length, and the fused pre-step's per-stream record.
#pragma once

#include "common.cuh"
#include "tc05.cuh"

namespace kws {

struct FrontendIo {
  PcmSource src;
  long S;
  int max_frames;           // row stride of mel_out in frames
  int groups;               // work items per stream = ceil(max_frames / the kernel's frames per item)
  int n_mel;
  float* mel_out;           // [S, max_frames, n_mel], or the recurrent kernel's fp16 operand (common.cuh) when tiled_out
  int tiled_out;
  int tile_chunks;          // tiled_out: chunks of 8 mels per half (kx / 8)
  int tile_split;           // tiled_out: the lo half (what the fp16 rounding lost) follows the hi half
  unsigned c_magic;         // ceil(2^32 / tile_chunks)
  unsigned q_magic;         // ceil(2^32 / (n_mel / 4)): i / Q == umulhi(i, q_magic) for i < 2^16
  int* nframes_out;         // [S] or null: frames per stream (fused pre-step, or streams of their own lengths)
  int fuse_pre;             // the server's pre-step (only with groups == 1 and int16 input): VAD, next tail
  FrontendPre pre;

  // samples of stream s the kernel transforms: its carried tail, then its body up to its own length under kLens
  template <bool kLens>
  __device__ __forceinline__ int total_len(long s, int head_len) const {
    return head_len + (kLens ? src.body_valid(s) : src.body_len);
  }
  // frames of stream s written to mel_out (the rest of its max_frames rows are zeros under kLens, untouched otherwise)
  __device__ __forceinline__ int frames(int total) const {
    const int n = frames_of(total);
    return n < max_frames ? n : max_frames;
  }

  // Frames [0, nfi) of a finished tile (row stride ld floats, n_mel bands per row) -> frames f0 .. f0 + nfi - 1 of
  // stream s, copied by threads t = 0 .. kThreads - 1.
  template <int kThreads>
  __device__ __forceinline__ void store_tile(const float* tile, int ld, long s, int f0, int nfi, int t) const {
    const int M = n_mel;
    const int total = nfi * M;
    if (tiled_out) {
      // the recurrent kernel's layer-0 operand (common.cuh): per frame, chunks of 8 mels as fp16 and (split) chunks of
      // what that rounding lost; the 16-byte piece (frame, chunk) of stream s sits between those of its 127 tile mates
      const int nc = tile_chunks;
      const int per_frame = tile_split ? 2 * nc : nc;
      uint4* dst = reinterpret_cast<uint4*>(mel_out) + ((s >> 7) * max_frames + f0) * static_cast<long>(per_frame) * 128 + (s & 127);
      const int pieces = nfi * nc;
      for (int i = t; i < pieces; i += kThreads) {
        const int f = nc == 1 ? i : static_cast<int>(__umulhi(static_cast<unsigned>(i), c_magic));   // i / nc, i < 2^16
        const int c = i - f * nc;
        const float* src = tile + f * ld + 8 * c;
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = 8 * c + j < M ? src[j] : 0.0f;
        uint4 hi, lo;
        tc::split_half8(v, &hi, &lo);
        dst[(f * per_frame + c) * 128] = hi;
        if (tile_split) dst[(f * per_frame + nc + c) * 128] = lo;
      }
    } else if ((M & 3) == 0 && (reinterpret_cast<uintptr_t>(mel_out) & 15) == 0) {
      // 16-byte pieces: chunk c (of Q) of frame f goes to row-major (s*n + f0 + f)*Q + c
      const int Q = M >> 2;
      float4* dst4 = reinterpret_cast<float4*>(mel_out) + (s * max_frames + f0) * static_cast<long>(Q);
      for (int i = t; i < (total >> 2); i += kThreads) {
        const int f = Q == 1 ? i : static_cast<int>(__umulhi(static_cast<unsigned>(i), q_magic));   // i / Q, i < 2^16
        const int c = i - f * Q;
        const float* src = tile + f * ld + 4 * c;
        dst4[i] = make_float4(src[0], src[1], src[2], src[3]);
      }
    } else {
      float* dst = mel_out + (s * max_frames + f0) * M;
      for (int i = t; i < total; i += kThreads) {
        const int f = i / M;
        dst[i] = tile[f * ld + (i - f * M)];
      }
    }
  }

  // frames [fa, fb) of stream s in mel_out (either layout) -> zero: the rows past a stream's length
  template <int kThreads>
  __device__ __forceinline__ void zero_rows(long s, int fa, int fb, int t) const {
    if (fb > max_frames) fb = max_frames;
    if (fa >= fb) return;
    if (tiled_out) {
      const int per_frame = tile_split ? 2 * tile_chunks : tile_chunks;
      uint4* dst = reinterpret_cast<uint4*>(mel_out) + ((s >> 7) * max_frames + fa) * static_cast<long>(per_frame) * 128 + (s & 127);
      for (int i = t; i < (fb - fa) * per_frame; i += kThreads) dst[static_cast<long>(i) * 128] = make_uint4(0u, 0u, 0u, 0u);
    } else {
      float* dst = mel_out + (s * max_frames + fa) * static_cast<long>(n_mel);
      for (int i = t; i < (fb - fa) * n_mel; i += kThreads) dst[i] = 0.0f;
    }
  }
};

int launch_frontend_tc(const kws_model* m, const FrontendIo& io, cudaStream_t st);   // frontend_tc.cu

}  // namespace kws
