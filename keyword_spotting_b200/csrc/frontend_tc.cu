// K1 on the tensor cores: framing + |rFFT_400| + mel as two tcgen05 GEMMs with a thread-local combination between.
//
// Replaces the same reference lines as frontend.cu (utils/stft.py:27-81, models/rnn_ctc.py:135-149; VAD and tail
// carry of detector.py:168-183 fused in for the streaming server) for int16 PCM.  Formulation (hop-block partial DFTs):
// a 400-sample frame at hop 160 is five 80-sample blocks, frame f = blocks 2f..2f+4, so
//     X_f(k) = sum_{j<5} w^(j k) P_{2f+j}(k),   w = e^(-2 pi i / 5),   P_b(k) = sum_{m<80} x[80 b + m] e^(-2 pi i m k / 400)
// and every block transform P_b is shared by the (up to three) frames that contain the block.
//
//   GEMM1  D[k, col] = sum_m T[k, m] * B[col, m]      (tcgen05.mma kind::f16, M = 128 lanes = frequencies k = 0..100,
//          two M tiles: T = cos and T = -sin; K = 80; N = 128 columns = 64 blocks x {x, (-1)^m x}).
//          The sign-alternated copy of a block gives the upper half of the spectrum on the SAME lane:
//          P_b(200 - k) = conj(P~_b(k)), so lane k owns frequencies k and 200 - k and needs no other lane's data.
//          The twiddles live in TENSOR MEMORY for the whole kernel (TS-form MMA, 160 columns), the PCM blocks in shared
//          memory (K-major canonical layout, two buffers).  Exactness: int16 x = x_hi + x_lo with x_hi = fp16(x) (exact
//          below 2048) and x_lo = x - x_hi (|x_lo| <= 8, exact), twiddle = T_hi + T_lo in fp16, product = T_hi*x_hi +
//          T_lo*x_hi + T_hi*x_lo accumulated in fp32; the dropped T_lo*x_lo is below 2^-23 of full scale and zero for
//          quiet signals, so the accuracy is that of an fp32 transform at every signal level.
//   combination (16 warps, thread = lane k x 8 frames): the 5-point twiddle sum for both of the lane's frequencies at
//          once in packed f32x2 (the coefficients depend on k mod 5 only and are the same for k and 200 - k up to
//          conjugation), magnitude, 8 frames = two 16-byte stores per frequency into the [bin][frame] magnitude
//          array in shared memory -- every step is thread-local: no shuffle, no transposition.
//   mel    (8 warps, lane = frame): mel[f, band] = sum_k basis[k, band] |X_f(k)| over the band's non-zero span, fp32
//          FMAs with broadcast weights and unit-stride magnitude reads, x 2^-15, [frame][band] tile -> 16-byte pieces.
//          (The projection was first a second tcgen05 GEMM -- basis^T x magnitudes, fp16 hi/lo in three MMAs; its 42
//          dependent N = 32 MMAs per item took ~170 cycles each and made the kernel 2x slower than the FFT one: see
//          profiles/r02_frontend_tc.md.)
//
// One CTA per SM, persistent over (stream, group of 30 frames) items; warp-specialised: 16 combination warps, 1 MMA
// issuer, 7 PCM loaders (int16 -> fp16 hi/lo operands, VAD sum, next tail), 8 mel/output warps; all hand-overs by mbarrier.
#include <cmath>
#include <cstdlib>
#include <vector>

#include <cuda_fp16.h>

#include "frontend_io.cuh"

namespace kws {

constexpr int kFtFrames = 30;                 // frames per work item
constexpr int kFtBlk = 80;                    // samples per block (hop / 2)
constexpr int kFtBlocks = 64;                 // blocks per work item (frames 0..29 use blocks 0..62)
constexpr int kFtWin = kFtBlocks * kFtBlk;    // 5120 samples
constexpr int kFtItemHop = kFtFrames * kHop;  // 4800 samples between the windows of consecutive items
constexpr int kFtPieces = kFtWin / 8;         // 16-byte pieces (8 samples) per window
constexpr int kFtRows = 2 * kFtBlocks;        // B1 rows: row 2b = block b, row 2b+1 = block b with (-1)^m
constexpr int kFtB1Lbo = 144;                 // bytes between K-adjacent core matrices (128 + 16: bank spread of the loader's stores)
constexpr int kFtB1Sbo = (kFtBlk / 8) * kFtB1Lbo;      // 1440 bytes between 8-row groups
constexpr int kFtB1Part = (kFtRows / 8) * kFtB1Sbo;    // 23040 bytes per operand part
constexpr int kFtMagStride = 36;              // floats per bin row of the magnitude array [bins][32 frames] (+4: conflict-free 16-byte stores)
constexpr int kFtMagRows = kBins + 7;         // band spans are padded to multiples of 8 bins (zero weights): rows 201..207 stay zero
constexpr int kFtMagFloats = kFtMagRows * kFtMagStride;
constexpr int kFtMaxMel = 64;
constexpr int kFtEpiWarps = 16;
constexpr int kFtMmaWarp = 16;
constexpr int kFtLoadWarp0 = 17, kFtLoadThreads = 7 * 32;      // the int16 -> fp16 hi/lo conversion is ~1.1 k warp-instructions per item
constexpr int kFtOutWarp0 = 24, kFtOutWarps = 8, kFtOutThreads = 32 * kFtOutWarps;   // the mel pass is latency-bound: 2 warps per scheduler
constexpr int kFtThreads = 32 * 32;
constexpr uint32_t kFtColA = 0;               // twiddles: [tile][part] x 40 columns (tile 0 cos, 1 -sin; part 0 hi, 1 lo)
// D_re: columns 160..287, D_im: 288..415.  One buffer: TMEM cannot hold two, and splitting an item's transforms into
// two N halves that are released separately was measured SLOWER -- a tcgen05.mma of this shape occupies the issue
// slot ~60 cycles whatever its N (64, 80 or 128), so 60 small MMAs cost twice what 30 big ones do.
constexpr uint32_t kFtColD = 160;
constexpr int kFtOutStride = 65;              // floats per frame row of the output tile (odd: conflict-free band writes)

enum { kFbBfull0 = 0, kFbBfull1, kFbBempty0, kFbBempty1, kFbDfull, kFbDempty, kFbMagFull0, kFbMagFull1, kFbMagEmpty0,
       kFbMagEmpty1, kFbNum };

struct FrontendTcParams : FrontendIo {
  const uint32_t* tw;       // [2 tiles][2 parts][128 lanes][40] packed fp16 pairs
  const int4* mel_seg;      // [n_mel] {first bin, bins (multiple of 8), offset into mel_w (multiple of 4), 0}
  const float* mel_w;       // the spans' weights, concatenated and zero-padded
  int mel_nw;               // floats in mel_w (multiple of 4)
  int vec_ok;               // int16 sources are 16-byte aligned with row strides % 8 == 0
};

__device__ __forceinline__ void ft_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
// Hand-overs on the critical cycle (D empty -> next block transforms -> D full -> combination): a tight
// test_wait poll for the single MMA warp, a try_wait with a short suspend hint for the 16 combination warps --
// the default try_wait suspends for an implementation-defined time and wakes late.
__device__ __forceinline__ void ft_spin(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = tc::smem_u32(bar);
  uint32_t ok = 0;
  for (uint32_t spins = 0; !ok; ++spins) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    if (spins > (1u << 28)) __trap();
  }
}
__device__ __forceinline__ void ft_wait_hint(uint64_t* bar, uint32_t parity, uint32_t ns) {
  const uint32_t addr = tc::smem_u32(bar);
  uint32_t ok = 0;
  for (uint32_t spins = 0; !ok; ++spins) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(addr), "r"(parity), "r"(ns)
        : "memory");
    if (spins > (1u << 26)) __trap();
  }
}
__device__ __forceinline__ float2 ft_sub2(float2 a, float2 b) { return __ffma2_rn(b, make_float2(-1.0f, -1.0f), a); }
__device__ __forceinline__ float ft_sqrt(float x) {
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// kLens: the streams have lengths of their own (p.src.lengths), as in frontend_kernel (frontend.cu); without them none of
// their handling is compiled in.
template <bool kLens>
__global__ void __launch_bounds__(kFtThreads, 1)
frontend_tc_kernel(const FrontendTcParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* sB1 = smem;                                            // [2 bufs][2 parts][kFtB1Part]
  float* sMag = reinterpret_cast<float*>(sB1 + 4 * kFtB1Part);          // [2 bufs][bins][kFtMagStride]
  float* sOut = sMag + 2 * kFtMagFloats;                                // [32][kFtOutStride]
  int4* sSeg = reinterpret_cast<int4*>(sOut + 32 * kFtOutStride);       // [kFtMaxMel]
  float* sW = reinterpret_cast<float*>(sSeg + kFtMaxMel);               // [mel_nw]
  int* sVad = reinterpret_cast<int*>(sW + p.mel_nw);                    // [2]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sVad + 2);               // [kFbNum]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kFbNum);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (warp == kFtMmaWarp) tc::tmem_alloc(tmem_slot, 512);
  if (tid == 0) {
    tc::mbar_init(&bars[kFbBfull0], kFtLoadThreads);
    tc::mbar_init(&bars[kFbBfull1], kFtLoadThreads);
    tc::mbar_init(&bars[kFbBempty0], 1);
    tc::mbar_init(&bars[kFbBempty1], 1);
    tc::mbar_init(&bars[kFbDfull], 1);
    tc::mbar_init(&bars[kFbDempty], 32 * kFtEpiWarps);
    tc::mbar_init(&bars[kFbMagFull0], 32 * kFtEpiWarps);
    tc::mbar_init(&bars[kFbMagFull1], 32 * kFtEpiWarps);
    tc::mbar_init(&bars[kFbMagEmpty0], kFtOutThreads);
    tc::mbar_init(&bars[kFbMagEmpty1], kFtOutThreads);
    tc::mbar_fence_init();
    sVad[0] = sVad[1] = 0;
  }
  for (int i = tid; i < p.n_mel; i += kFtThreads) sSeg[i] = __ldg(p.mel_seg + i);
  for (int i = tid; i < p.mel_nw; i += kFtThreads) sW[i] = __ldg(p.mel_w + i);
  for (int i = tid; i < 2 * kFtMagFloats; i += kFtThreads) sMag[i] = 0.0f;       // rows 201..207 are never written again
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = *tmem_slot;

  if (warp < 4) {                     // the twiddles -> TMEM: lane 32*warp + lane owns row k of both tiles, hi and lo
    const uint32_t row = tmem + (static_cast<uint32_t>(32 * warp) << 16) + kFtColA;
#pragma unroll 1
    for (int tp = 0; tp < 4; ++tp) {
      const uint32_t* src = p.tw + (static_cast<long>(tp) * 128 + 32 * warp + lane) * 40;
      uint32_t v[16];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = __ldg(src + 16 * h + j);
        tc::st16(row + 40 * tp + 16 * h, v);
      }
      uint32_t w[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) w[j] = __ldg(src + 32 + j);
      tc::st8(row + 40 * tp + 32, w);
    }
    tc::wait_st();
  }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();

  const long items = p.S * p.groups;
  const long n_mine = (items - blockIdx.x + gridDim.x - 1) / gridDim.x;       // items of this CTA
  const int M = p.n_mel;

  // per-item geometry, the same in every role
  auto item_of = [&](long i) -> long { return blockIdx.x + i * static_cast<long>(gridDim.x); };
  auto stream_of = [&](long item) -> long { return p.groups == 1 ? item : item / p.groups; };

  // Registers: 1024 threads are launched at 64 each, the combination role needs ~76 (at 64 it spilled a dozen values per
  // item, and a spill reload is an L2 round trip next to 170 KB of shared memory).  setmaxnreg moves 16 registers per
  // thread from warpgroups 4-7 (issuer, loaders, mel) to warpgroups 0-3; the instruction is warpgroup-wide and the pool
  // of a CTA is what it was launched with, so the two sides must balance exactly: 512 x (+16) = 512 x (-16).
  // (one instruction at the head of every role's branch: the compiler budgets a region by the setmaxnreg that dominates it)
  if (warp == kFtMmaWarp) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 48;");
    // ================================================================ MMA issuer
    const uint64_t b1desc = tc::smem_desc(tc::smem_u32(sB1), kFtB1Lbo, kFtB1Sbo);
    // an item's block transforms: Re tile, then Im tile.  The issuing warp shares its scheduler with seven others and
    // a tcgen05.mma holds the issue slot ~60 cycles: fully unrolled, every operand address in uniform registers.
    const uint32_t idesc = tc::idesc_f16(128, 128);
    // (issued from one elect.sync region: back-to-back UTCHMMA -- under a `lane == 0` predicate ptxas wraps every MMA in
    // a six-instruction loop over the active lanes)
    auto gemm1 = [&](uint64_t bH, uint64_t bL, uint64_t* bar_d, uint64_t* bar_b) {
      if (tc::elect_one()) {
#pragma unroll
        for (int tile = 0; tile < 2; ++tile) {
          const uint32_t d = tmem + kFtColD + 128 * tile;
          const uint32_t a_hi = tmem + kFtColA + 40 * (2 * tile), a_lo = a_hi + 40;
#pragma unroll
          for (int k16 = 0; k16 < kFtBlk / 16; ++k16) {
            const uint64_t step = static_cast<uint64_t>(k16 * ((2 * kFtB1Lbo) >> 4));
            tc::mma_ts(d, a_hi + 8 * k16, bH + step, idesc, k16 > 0);
            tc::mma_ts(d, a_hi + 8 * k16, bL + step, idesc, true);
            tc::mma_ts(d, a_lo + 8 * k16, bH + step, idesc, true);
          }
        }
        tc::commit(bar_d);
        tc::commit(bar_b);
      }
    };
    for (long i = 0; i < n_mine; ++i) {
      const int buf = static_cast<int>(i & 1);
      ft_spin(&bars[kFbBfull0 + buf], static_cast<uint32_t>((i >> 1) & 1));
      if (i > 0) ft_spin(&bars[kFbDempty], static_cast<uint32_t>((i - 1) & 1));
      tc::fence_after_sync();
      // (the buffer index is loop-carried, which the compiler cannot prove warp-uniform: branch on it so that every
      // descriptor inside is derived from kernel constants and stays in uniform registers -- no per-MMA broadcast loop)
      constexpr uint64_t kPart = static_cast<uint64_t>(kFtB1Part >> 4);
      if (buf == 0) gemm1(b1desc, b1desc + kPart, &bars[kFbDfull], &bars[kFbBempty0]);
      else gemm1(b1desc + 2 * kPart, b1desc + 3 * kPart, &bars[kFbDfull], &bars[kFbBempty1]);
    }
  } else if (warp >= kFtLoadWarp0 && warp < kFtOutWarp0) {
    // ================================================================ PCM loaders: int16 -> (x_hi, x_lo) fp16 operands
    asm volatile("setmaxnreg.dec.sync.aligned.u32 48;");
    const int ltid = tid - 32 * kFtLoadWarp0;
    for (long i = 0; i < n_mine; ++i) {
      const long item = item_of(i);
      const long s = stream_of(item);
      const int g = static_cast<int>(item - s * p.groups);
      const int buf = static_cast<int>(i & 1);
      const int head_len = p.src.head_len ? p.src.head_len[s] : 0;
      const int total_len = p.total_len<kLens>(s, head_len);
      // samples staged from PCM: none for an item past the stream's last frame (its rows are zeros), otherwise those
      // below the stream's length -- the piece that straddles it goes element by element, the rest stage as zeros
      const int ld_len = kLens && g * kFtFrames >= frames_of(total_len) ? 0 : total_len;
      const int q0 = g * kFtItemHop;
      const int16_t* body = static_cast<const int16_t*>(p.src.body) + s * p.src.ld_body - head_len;   // indexed by stream sample
      const int16_t* head = p.src.head ? p.src.head + s * p.src.ld_head : nullptr;
      const bool fast = p.vec_ok && (head_len & 7) == 0;
      // server pre-step (detector.py:168-183)
      const int keep = tail_keep(total_len);
      const int start = total_len - keep;
      int16_t* tnext = p.fuse_pre ? p.pre.tail_next + s * 400 : nullptr;
      const bool tail_fast = p.fuse_pre && ((start | keep) & 7) == 0 && (reinterpret_cast<uintptr_t>(p.pre.tail_next) & 15) == 0;
      const int n_pieces = p.fuse_pre ? kFtPieces + 10 : kFtPieces;       // the fused chunk may reach 5199 samples
      // every piece this thread owns is requested before anything is waited for: one HBM latency per item, not seven
      constexpr int kRounds = (kFtPieces + 10 + kFtLoadThreads - 1) / kFtLoadThreads;
      uint4 pre[kRounds];
#pragma unroll
      for (int rd = 0; rd < kRounds; ++rd) {
        const int pc = ltid + kFtLoadThreads * rd;
        const int q = q0 + 8 * pc;
        pre[rd] = make_uint4(0u, 0u, 0u, 0u);
        if (pc < n_pieces && fast && q + 8 <= ld_len)
          pre[rd] = __ldg(reinterpret_cast<const uint4*>((q < head_len ? head : body) + q));
      }
      if (i >= 2) ft_wait_hint(&bars[kFbBempty0 + buf], static_cast<uint32_t>(((i >> 1) + 1) & 1), 200);
      unsigned char* dstS = sB1 + (buf * 2 + 0) * kFtB1Part;
      unsigned char* dstU = sB1 + (buf * 2 + 1) * kFtB1Part;
      float vadf = 0.0f;
#pragma unroll
      for (int rd = 0; rd < kRounds; ++rd) {
        const int pc = ltid + kFtLoadThreads * rd;
        if (pc >= n_pieces) break;
        const int q = q0 + 8 * pc;
        uint4 v = pre[rd];
        if (q < ld_len && !(fast && q + 8 <= ld_len)) {                   // unaligned rows / the ragged end: element by element
          unsigned e[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            int x = 0;
            if (q + j < head_len) x = head[q + j];
            else if (q + j < ld_len) x = body[q + j];
            e[j] = static_cast<unsigned>(x) & 0xffffu;
          }
          v = make_uint4(e[0] | (e[1] << 16), e[2] | (e[3] << 16), e[4] | (e[5] << 16), e[6] | (e[7] << 16));
        }
        const unsigned w[4] = {v.x, v.y, v.z, v.w};
        float f[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          f[2 * j] = static_cast<float>(static_cast<short>(w[j] & 0xffffu));
          f[2 * j + 1] = static_cast<float>(static_cast<short>(w[j] >> 16));
        }
        if (p.fuse_pre && q < total_len) {
          // VAD on the NEW samples (detector.py:168): |x| summed in fp32, exact (integers far below 2^24)
          if (q >= head_len) {
            vadf += ((fabsf(f[0]) + fabsf(f[1])) + (fabsf(f[2]) + fabsf(f[3]))) + ((fabsf(f[4]) + fabsf(f[5])) + (fabsf(f[6]) + fabsf(f[7])));
          } else if (q + 8 > head_len) {              // a piece that straddles the carried tail (unaligned tails only)
#pragma unroll
            for (int j = 0; j < 8; ++j) vadf += q + j >= head_len ? fabsf(f[j]) : 0.0f;
          }
          if (q + 8 > start) {                                            // next carried tail
            if (tail_fast) {
              *reinterpret_cast<uint4*>(tnext + (q - start)) = v;         // start, keep, q multiples of 8: whole pieces
            } else {
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const int idx = q + j - start;
                if (idx >= 0 && q + j < total_len)
                  tnext[idx] = static_cast<int16_t>((j & 1) ? (w[j >> 1] >> 16) : (w[j >> 1] & 0xffffu));
              }
            }
          }
        }
        if (pc < kFtPieces) {
          uint4 oS, oU, oSa, oUa;
          unsigned* os = &oS.x; unsigned* ou = &oU.x; unsigned* osa = &oSa.x; unsigned* oua = &oUa.x;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            // x = x_hi + x_lo: x_hi = fp16(x) (11 significant bits; exact below 2048), x_lo = x - x_hi (|x_lo| <= 8, exact)
            const __half2 hh = __floats2half2_rn(f[2 * j], f[2 * j + 1]);
            const float2 hf = __half22float2(hh);
            const __half2 ll = __floats2half2_rn(f[2 * j] - hf.x, f[2 * j + 1] - hf.y);
            os[j] = *reinterpret_cast<const unsigned*>(&hh);
            ou[j] = *reinterpret_cast<const unsigned*>(&ll);
            oua[j] = ou[j] ^ 0x80000000u;                                 // (-1)^m: the odd sample of the pair
            osa[j] = os[j] ^ 0x80000000u;
          }
          const int b = (pc * 52429) >> 19, c = pc - 10 * b;              // pc / 10 for pc < 81920
          const int off = ((2 * b) >> 3) * kFtB1Sbo + c * kFtB1Lbo + ((2 * b) & 7) * 16;
          *reinterpret_cast<uint4*>(dstS + off) = oS;
          *reinterpret_cast<uint4*>(dstS + off + 16) = oSa;
          *reinterpret_cast<uint4*>(dstU + off) = oU;
          *reinterpret_cast<uint4*>(dstU + off + 16) = oUa;
        }
      }
      if (p.fuse_pre) {
        const int vad = __reduce_add_sync(0xffffffffu, static_cast<int>(vadf));
        if (lane == 0) atomicAdd(&sVad[buf], vad);
        asm volatile("bar.sync 2, 224;" ::: "memory");
        if (ltid == 0) {
          p.pre.record(s, sVad[buf], p.frames(total_len), keep, p.nframes_out);
          sVad[buf] = 0;
        }
      }
      tc::fence_proxy_async();
      ft_arrive(&bars[kFbBfull0 + buf]);
    }
  } else if (warp >= kFtOutWarp0) {
    // ================================================================ mel projection + output: lane = frame
    asm volatile("setmaxnreg.dec.sync.aligned.u32 48;");
    const int otid = tid - 32 * kFtOutWarp0;
    const int q = warp - kFtOutWarp0;
    for (long i = 0; i < n_mine; ++i) {
      const long item = item_of(i);
      const long s = stream_of(item);
      const int g = static_cast<int>(item - s * p.groups);
      const int buf = static_cast<int>(i & 1);
      const int head_len = p.src.head_len ? p.src.head_len[s] : 0;
      const int nfr = p.frames(p.total_len<kLens>(s, head_len));
      const int f0 = g * kFtFrames;
      const int nfi = max(0, min(nfr - f0, kFtFrames));
      if (kLens && p.nframes_out && g == 0 && otid == 0) p.nframes_out[s] = nfr;
      ft_wait_hint(&bars[kFbMagFull0 + buf], static_cast<uint32_t>((i >> 1) & 1), 200);
      // bands q, q+8, ...: eight bins per trip (spans are zero-padded to multiples of 8): the eight magnitude loads
      // (32 consecutive floats each) and the two broadcast weight loads are independent, four accumulators
      const float* mcol = sMag + buf * kFtMagFloats + lane;
#pragma unroll 1
      for (int band = q; band < M; band += kFtOutWarps) {
        const int4 seg = sSeg[band];
        const float4* wp = reinterpret_cast<const float4*>(sW + seg.z);
        const float* mp = mcol + seg.x * kFtMagStride;
        float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
#pragma unroll 1
        for (int j = 0; j < seg.y; j += 8) {
          const float4 w0 = wp[j >> 2], w1 = wp[(j >> 2) + 1];
          const float m0 = mp[(j + 0) * kFtMagStride], m1 = mp[(j + 1) * kFtMagStride], m2 = mp[(j + 2) * kFtMagStride],
                      m3 = mp[(j + 3) * kFtMagStride], m4 = mp[(j + 4) * kFtMagStride], m5 = mp[(j + 5) * kFtMagStride],
                      m6 = mp[(j + 6) * kFtMagStride], m7 = mp[(j + 7) * kFtMagStride];
          a0 = fmaf(w0.x, m0, a0);
          a1 = fmaf(w0.y, m1, a1);
          a2 = fmaf(w0.z, m2, a2);
          a3 = fmaf(w0.w, m3, a3);
          a0 = fmaf(w1.x, m4, a0);
          a1 = fmaf(w1.y, m5, a1);
          a2 = fmaf(w1.z, m6, a2);
          a3 = fmaf(w1.w, m7, a3);
        }
        if (lane < kFtFrames) sOut[lane * kFtOutStride + band] = ((a0 + a1) + (a2 + a3)) * 3.0517578125e-05f;   // 2^-15 (detector.py:40-43)
      }
      ft_arrive(&bars[kFbMagEmpty0 + buf]);          // this thread's magnitude reads are done
      asm volatile("bar.sync 3, 256;" ::: "memory");
      p.store_tile<kFtOutThreads>(sOut, kFtOutStride, s, f0, nfi, otid);
      if (kLens) p.zero_rows<kFtOutThreads>(s, f0 + nfi, f0 + kFtFrames, otid);   // the item's frames past the stream's length
      asm volatile("bar.sync 3, 256;" ::: "memory");
    }
  } else {
    // ================================================================ combination: lane k (and 200 - k) x 8 frames
    asm volatile("setmaxnreg.inc.sync.aligned.u32 80;");
    const int q = warp & 3, F = warp >> 2;
    const int k = 32 * q + lane;
    const uint32_t lane_sel = static_cast<uint32_t>(32 * q) << 16;
    const int r = k % 5;
    // w^(j k) = c_j - i s_j, c_j = cos(2 pi j r / 5), s_j = sin(2 pi j r / 5); c_4 = c_1, c_3 = c_2, s_4 = -s_1, s_3 = -s_2
    const float kc1 = 0.30901699437494745f, kc2 = -0.8090169943749473f, ks1 = 0.9510565162951535f, ks2 = 0.5877852522924732f;
    // (cos, sin)(2 pi r / 5) and (cos, sin)(4 pi r / 5) for r = 0..4
    const float c1s = r == 0 ? 1.0f : ((r == 1 || r == 4) ? kc1 : kc2);
    const float s1s = r == 0 ? 0.0f : (r == 1 ? ks1 : (r == 2 ? ks2 : (r == 3 ? -ks2 : -ks1)));
    const float c2s = r == 0 ? 1.0f : ((r == 2 || r == 3) ? kc1 : kc2);
    const float s2s = r == 0 ? 0.0f : (r == 1 ? ks2 : (r == 2 ? -ks1 : (r == 3 ? ks1 : -ks2)));
    const float2 c1 = make_float2(c1s, c1s), c2 = make_float2(c2s, c2s), s1 = make_float2(s1s, s1s), s2 = make_float2(s2s, s2s);
    const float2 ns1 = make_float2(-s1s, -s1s), ns2 = make_float2(-s2s, -s2s);
    float* mag_k = sMag + k * kFtMagStride + 8 * F;                 // bin k, frames 8F..8F+7
    float* mag_u = sMag + (200 - k) * kFtMagStride + 8 * F;         // bin 200 - k
    const uint32_t dre = tmem + lane_sel + kFtColD + 32 * F, dim = dre + 128;

    for (long i = 0; i < n_mine; ++i) {
      ft_wait_hint(&bars[kFbDfull], static_cast<uint32_t>(i & 1), 100);
      tc::fence_after_sync();
      float2 mg[8];                                   // (|X_f(k)|, |X_f(200-k)|) of frames 8F .. 8F+7
      // TMEM reads run at ~64 B/clk per SM and are what this role is bound by: every column is read exactly once.
      // frames 8F+4sub .. +3 use blocks 16F+8sub .. +10 (two columns per block: x, (-1)^m x):
      //   sub 0: columns 0..23 of the warp's window (blocks 0..11);  sub 1: keeps blocks 8..11, reads columns 24..39
      uint32_t re[24], im[24];
#pragma unroll
      for (int sub = 0; sub < 2; ++sub) {
        if (sub == 0) {
          uint32_t a16[16], a8[8], b16[16], b8[8];
          tc::ld16(dre, a16);
          tc::ld8(dre + 16, a8);
          tc::ld16(dim, b16);
          tc::ld8(dim + 16, b8);
          tc::wait_ld();
#pragma unroll
          for (int j = 0; j < 16; ++j) { re[j] = a16[j]; im[j] = b16[j]; }
#pragma unroll
          for (int j = 0; j < 8; ++j) { re[16 + j] = a8[j]; im[16 + j] = b8[j]; }
        } else {
          uint32_t a16[16], b16[16];
          tc::ld16(dre + 24, a16);
          tc::ld16(dim + 24, b16);
#pragma unroll
          for (int j = 0; j < 8; ++j) { re[j] = re[16 + j]; im[j] = im[16 + j]; }
          tc::wait_ld();
#pragma unroll
          for (int j = 0; j < 16; ++j) { re[8 + j] = a16[j]; im[8 + j] = b16[j]; }
          tc::fence_before_sync();                    // every TMEM read of this item is done: the half may be overwritten
          ft_arrive(&bars[kFbDempty]);
        }
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const int b0 = 2 * t;
          auto P = [&](int b) { return make_float2(__uint_as_float(re[2 * b]), __uint_as_float(re[2 * b + 1])); };
          auto Q = [&](int b) { return make_float2(__uint_as_float(im[2 * b]), __uint_as_float(im[2 * b + 1])); };
          const float2 s14r = __fadd2_rn(P(b0 + 1), P(b0 + 4)), d14r = ft_sub2(P(b0 + 1), P(b0 + 4));
          const float2 s23r = __fadd2_rn(P(b0 + 2), P(b0 + 3)), d23r = ft_sub2(P(b0 + 2), P(b0 + 3));
          const float2 s14i = __fadd2_rn(Q(b0 + 1), Q(b0 + 4)), d14i = ft_sub2(Q(b0 + 1), Q(b0 + 4));
          const float2 s23i = __fadd2_rn(Q(b0 + 2), Q(b0 + 3)), d23i = ft_sub2(Q(b0 + 2), Q(b0 + 3));
          float2 xr = __ffma2_rn(c1, s14r, P(b0));
          xr = __ffma2_rn(c2, s23r, xr);
          xr = __ffma2_rn(s1, d14i, xr);
          xr = __ffma2_rn(s2, d23i, xr);
          float2 xi = __ffma2_rn(c1, s14i, Q(b0));
          xi = __ffma2_rn(c2, s23i, xi);
          xi = __ffma2_rn(ns1, d14r, xi);
          xi = __ffma2_rn(ns2, d23r, xi);
          const float2 m2 = __ffma2_rn(xi, xi, __fmul2_rn(xr, xr));
          mg[4 * sub + t] = make_float2(ft_sqrt(m2.x), ft_sqrt(m2.y));
        }
      }
      const int mbuf = static_cast<int>(i & 1);
      if (i >= 2) ft_wait_hint(&bars[kFbMagEmpty0 + mbuf], static_cast<uint32_t>(((i >> 1) + 1) & 1), 200);
      if (k <= 100) {                                 // lanes 101..127 carry zero twiddle rows (nothing to store)
        float* dk = mag_k + mbuf * kFtMagFloats;
        *reinterpret_cast<float4*>(dk) = make_float4(mg[0].x, mg[1].x, mg[2].x, mg[3].x);
        *reinterpret_cast<float4*>(dk + 4) = make_float4(mg[4].x, mg[5].x, mg[6].x, mg[7].x);
        if (k < 100) {                                // bin 100 is its own mirror
          float* du = mag_u + mbuf * kFtMagFloats;
          *reinterpret_cast<float4*>(du) = make_float4(mg[0].y, mg[1].y, mg[2].y, mg[3].y);
          *reinterpret_cast<float4*>(du + 4) = make_float4(mg[4].y, mg[5].y, mg[6].y, mg[7].y);
        }
      }
      ft_arrive(&bars[kFbMagFull0 + mbuf]);
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == kFtMmaWarp) tc::tmem_dealloc(tmem, 512);
}

static size_t frontend_tc_smem_bytes(int mel_nw) {
  return static_cast<size_t>(4) * kFtB1Part + sizeof(float) * (2 * kFtMagFloats + 32 * kFtOutStride + mel_nw) +
         sizeof(int4) * kFtMaxMel + sizeof(int) * 2 + sizeof(uint64_t) * kFbNum + 16;
}

// Tables of the tensor-core front end for a basis [201, M]: twiddles as TMEM rows (fp16 hi / lo), and the non-zero span
// of every mel band with its weights.
int build_frontend_tc_tables(kws_model* m, const float* basis) {
  const int M = m->cfg.n_mel;
  m->fe_tc.ready = false;
  if (M > kFtMaxMel) return KWS_OK;                        // wider filterbanks stay on the FFT kernel
  std::vector<uint32_t> tw(static_cast<size_t>(4) * 128 * 40, 0u);
  for (int tile = 0; tile < 2; ++tile)
    for (int k = 0; k <= 100; ++k)
      for (int mm = 0; mm < kFtBlk; ++mm) {
        const double a = 2.0 * M_PI * static_cast<double>((mm * k) % 400) / 400.0;
        const double v = tile == 0 ? std::cos(a) : -std::sin(a);
        const __half hi = __float2half_rn(static_cast<float>(v));
        const __half lo = __float2half_rn(static_cast<float>(v - static_cast<double>(__half2float(hi))));
        const unsigned short hb = *reinterpret_cast<const unsigned short*>(&hi), lb = *reinterpret_cast<const unsigned short*>(&lo);
        uint32_t& wh = tw[(static_cast<size_t>(2 * tile + 0) * 128 + k) * 40 + mm / 2];
        uint32_t& wl = tw[(static_cast<size_t>(2 * tile + 1) * 128 + k) * 40 + mm / 2];
        wh |= static_cast<uint32_t>(hb) << (16 * (mm & 1));
        wl |= static_cast<uint32_t>(lb) << (16 * (mm & 1));
      }
  // the non-zero span of every band (exact for any basis: zeros inside a span are multiplied like any weight)
  std::vector<int4> seg(M);
  std::vector<float> wts;
  for (int band = 0; band < M; ++band) {
    int lo = -1, hi = -1;
    for (int k = 0; k < kBins; ++k)
      if (basis[static_cast<size_t>(k) * M + band] != 0.0f) {
        if (lo < 0) lo = k;
        hi = k;
      }
    if (lo < 0) lo = hi = 0;                               // an all-zero band: zero weights
    const int n = (hi - lo + 1 + 7) / 8 * 8;               // padded to whole trips of the kernel's loop (zero weights)
    seg[band] = make_int4(lo, n, static_cast<int>(wts.size()), 0);
    for (int j = 0; j < n; ++j) wts.push_back(lo + j <= hi ? basis[static_cast<size_t>(lo + j) * M + band] : 0.0f);
  }
  m->fe_tc.mel_nw = static_cast<int>(wts.size());
  KWS_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&m->fe_tc.tw), tw.size() * sizeof(uint32_t)));
  KWS_CUDA_OK(cudaMemcpy(m->fe_tc.tw, tw.data(), tw.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
  KWS_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&m->fe_tc.mel_seg), seg.size() * sizeof(int4)));
  KWS_CUDA_OK(cudaMemcpy(m->fe_tc.mel_seg, seg.data(), seg.size() * sizeof(int4), cudaMemcpyHostToDevice));
  KWS_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&m->fe_tc.mel_w), wts.size() * sizeof(float)));
  KWS_CUDA_OK(cudaMemcpy(m->fe_tc.mel_w, wts.data(), wts.size() * sizeof(float), cudaMemcpyHostToDevice));
  m->fe_tc.ready = true;
  return KWS_OK;
}

void free_frontend_tc_tables(kws_model* m) {
  cudaFree(m->fe_tc.tw);
  cudaFree(m->fe_tc.mel_seg);
  cudaFree(m->fe_tc.mel_w);
  m->fe_tc = FrontendTcTables();
}

// Which front end serves this launch.  The FFT kernel (frontend.cu) is the default: on B200 the two run at the same
// speed (2.4 ms for 131,072 x 30 frames) and the FFT is the more accurate one (1e-7 vs 3e-7 of the float64 spectrum).
// The tensor-core kernel is selected per model (kws_model_set_frontend) or with KWS_FRONTEND=tc in the environment; it
// serves int16 PCM only (arbitrary floats have no exact two-term fp16 split) and filterbanks of up to 64 bands.
bool frontend_uses_tc(const kws_model* m, int pcm_dtype) {
  return m->frontend == KWS_FRONTEND_TC && m->fe_tc.ready && pcm_dtype == KWS_PCM_I16;
}

int default_frontend() {
  static const int choice = [] {
    const char* e = std::getenv("KWS_FRONTEND");
    return e && e[0] == 't' ? KWS_FRONTEND_TC : KWS_FRONTEND_FFT;
  }();
  return choice;
}

int frontend_tc_item_frames() { return kFtFrames; }

int launch_frontend_tc(const kws_model* m, const FrontendIo& io, cudaStream_t st) {
  FrontendTcParams p{io};
  p.tw = m->fe_tc.tw;
  p.mel_seg = reinterpret_cast<const int4*>(m->fe_tc.mel_seg);
  p.mel_w = m->fe_tc.mel_w;
  p.mel_nw = m->fe_tc.mel_nw;
  p.vec_ok = (reinterpret_cast<uintptr_t>(io.src.body) % 16 == 0 && io.src.ld_body % 8 == 0 &&
              reinterpret_cast<uintptr_t>(io.src.head) % 16 == 0 && io.src.ld_head % 8 == 0) ? 1 : 0;
  auto kernel = io.src.lengths ? frontend_tc_kernel<true> : frontend_tc_kernel<false>;
  const size_t smem = frontend_tc_smem_bytes(p.mel_nw);
  KWS_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const long items = io.S * io.groups;
  const long blocks = items < sm_count() ? items : sm_count();
  kernel<<<static_cast<unsigned>(blocks), kFtThreads, smem, st>>>(p);
  KWS_LAUNCH_OK("frontend_tc_kernel");
  return KWS_OK;
}

}  // namespace kws
