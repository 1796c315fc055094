// K1 -- fused framing + 400-point real DFT magnitude + mel projection (+ the server's per-chunk pre-step).
//
// Replaces, in one pass over the PCM and without materialising frames or spectra:
//   tf_frame(signal, 400, 160)            utils/stft.py:27-81   (rect window, no padding)
//   tf.abs(tf.spectral.rfft(frames,[400])) models/rnn_ctc.py:137
//   tf.matmul(linearspec, mel_basis)       models/rnn_ctc.py:139-149
// and, when launched by the streaming server for a chunk that fits one work item, also
//   vad(data, 30)                          utils/basic_vad.py:17-18, detector.py:168
//   tail carry (len-400)%160+240           detector.py:179-183
// so the chunk's PCM is read from HBM exactly once.
//
// Work item = (stream, group of 16 consecutive frame PAIRS = 32 frames) handled by one 320-thread CTA:
// thread t = 20*pair + column owns one DFT-20 column of its pair in both stages of the packed-real 20x20 FFT
// (fft400.cuh).  The item's PCM (5360 samples) is staged once in shared memory as fp32 with coalesced 16-byte
// loads; every 320-sample block is skewed by 20 floats so that the 32 lanes of a warp -- which straddle two
// pairs -- read 32 distinct banks.  int16 PCM is fetched four samples per load (8 bytes) and the NEXT work item's
// loads are issued before the mel projection of the current one, so their latency is hidden behind it.  int16
// samples are transformed unscaled (the DFT is linear); 2^-15 and the 1/2 of the two-for-one untangling are applied
// once per mel band.  Magnitudes go to shared memory transposed ([bin][frame]) so that the mel projection runs
// with lane = frame and warp-uniform weights: the non-zero part of the basis is cut at model creation into "quads"
// (4 consecutive bins of one band, build_mel_quads), whole bands are dealt to the 10 warps so that every warp gets
// the same number of quads (longest-band-first), and the kernel runs one flat, branch-free loop over its quads
// (~2*201 FMAs per frame for a triangular filterbank, exact for any dense basis) with broadcast weight reads and
// conflict-free magnitude reads; the [32, M] result tile leaves as one contiguous block.  Persistent grid:
// (resident CTAs per SM) x 148 SMs, grid-stride over work items.
#include <algorithm>
#include <cstring>
#include <vector>

#include "fft400.cuh"
#include "frontend_io.cuh"

namespace kws {

using fft::cpx;

constexpr int kFePairs = 16;                         // frame pairs per work item
constexpr int kFeThreads = kFePairs * fft::kR;       // 320
constexpr int kFeWarps = kFeThreads / 32;            // 10
constexpr int kFeItemFrames = 2 * kFePairs;          // 32
constexpr int kFeBlock = 2 * kHop;                   // 320 samples between consecutive pairs
constexpr int kFeSkew = 20;                          // floats of skew per 320-sample block
constexpr int kFeWinSamples = kFePairs * kFeBlock + (kFft - kHop);       // 5360
constexpr int kFeWinRounds = (kFeWinSamples + kFeThreads - 1) / kFeThreads;   // 17
constexpr int kFeQuadRounds = (kFeWinSamples + 4 * kFeThreads - 1) / (4 * kFeThreads);      // 5 (int16: 4 samples per load)
constexpr int kFeLastQuads = (kFeWinSamples - 4 * kFeThreads * (kFeQuadRounds - 1)) / 4;    // 60 threads in the last round
static_assert(kFeWinSamples % 4 == 0 && kFeBlock % 4 == 0, "quads must not straddle a skew boundary");
constexpr int kFeQuadSmemMax = 512;                  // quads kept in shared memory (32 B each, keeps 2 CTAs per SM); more -> read from global
constexpr int kFeItemHop = kFePairs * kFeBlock;      // 5120 samples between consecutive items of a stream
constexpr int kFeMagStride = 66;                     // floats per row of the transposed magnitudes [102 bin pairs][32 slots][2] (+2 pad)
// the window (5360 samples + skew) and the transposed magnitudes share one region: the window is dead after stage 1
constexpr int kFeWinFloats = kFeWinRounds * (kFeBlock + kFeSkew);        // 5780 (position tid + 340*round)
constexpr int kFeMagRows = (fft::kBins + 3) / 2;     // quads are 4 bins from an even bin: bins 201..203 stay zero
constexpr int kFeMagFloats = kFeMagRows * kFeMagStride;
constexpr int kFeMagLive = (fft::kBins / 2) * kFeMagStride;   // rows below hold only written bins (0..199)
constexpr int kFeRegionFloats = kFeMagFloats > kFeWinFloats ? kFeMagFloats : kFeWinFloats;
static_assert(kFeWinFloats <= kFeMagLive, "the window must not reach the rows that hold the zero bins");
static_assert((kFeRegionFloats * 4) % 16 == 0, "mel quads follow the region and are read as float4");

struct FrontendParams : FrontendIo {
  const cpx* twiddle;       // [20*52] periodic k2-major table (fft::kTwSlots)
  const MelQuad* mel_q;     // [10 warps][quads_per_warp] (common.cuh)
  int mel_qpw;              // quads per warp (even)
  int vec_ok;               // int16 sources are 8-byte aligned with row strides % 4 == 0
  float mag_scale;          // 0.5 * (int16 input ? 2^-15 : 1), applied to the finished band sums
};

// Transposed magnitudes: bin k of frame slot sl sits at (k/2)*66 + 2*sl + (k&1), so the mel projection (lane = slot)
// reads two consecutive bins with one conflict-free 64-bit load.  Frame slot of frame fr of pair p: chosen so that the
// 32 lanes of a warp in the untangle phase (consecutive columns k2 of adjacent pairs, same k1) hit 32 distinct banks:
// bank = (k + 2*slot) mod 32 must advance by 20 per pair, i.e. slot = 10*p mod 16; pairs 8..15 take the upper 16
// slots.  The 2 x 16 frames fill the 32 slots exactly once.
__device__ __forceinline__ int mag_slot(int pair, int fr) { return ((10 * pair) & 15) + 16 * (pair >> 3) + fr; }
// inverse: slot -> frame index 2*pair + fr within the item  (5*5 = 25 = 1 mod 8)
__device__ __forceinline__ int slot_frame(int slot) {
  const int pair = ((5 * ((slot & 15) >> 1)) & 7) + 8 * (slot >> 4);
  return 2 * pair + (slot & 1);
}
__device__ __forceinline__ int mag_index(int bin, int slot) { return (bin >> 1) * kFeMagStride + 2 * slot + (bin & 1); }

// four int16 samples of one 8-byte load -> floats (exact)
__device__ __forceinline__ float4 quad_to_float(uint2 q) {
  return make_float4(static_cast<float>(static_cast<short>(q.x & 0xffffu)), static_cast<float>(static_cast<short>(q.x >> 16)),
                     static_cast<float>(static_cast<short>(q.y & 0xffffu)), static_cast<float>(static_cast<short>(q.y >> 16)));
}

// kLens: the streams have lengths of their own (p.src.lengths): zero-fill past each length, skip items past each stream's
// last frame, write the frame counts.  Without them none of that is compiled in (the streaming server's path, and every
// equal-length forward).
template <bool kQuadsInSmem, bool kLens>
__global__ void __launch_bounds__(kFeThreads, 2)
frontend_kernel(const FrontendParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cpx* twp = reinterpret_cast<cpx*>(smem_raw);                      // [1040]
  cpx* buf = twp + fft::kTwSlots;                                   // [16][420]; later the [32][M] output tile
  float* win = reinterpret_cast<float*>(buf + kFePairs * fft::kBufSlots);   // window, later magnitudes [102][66]
  int* red = reinterpret_cast<int*>(win + kFeRegionFloats);         // [16] block reduction scratch
  MelQuad* s_q = reinterpret_cast<MelQuad*>(red + 16);              // [10][qpw]   (only when kQuadsInSmem)

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < fft::kTwSlots; i += kFeThreads) twp[i] = p.twiddle[i];
  if (kQuadsInSmem) {
    const int n16 = kFeWarps * p.mel_qpw * static_cast<int>(sizeof(MelQuad) / 16);
    for (int i = tid; i < n16; i += kFeThreads) reinterpret_cast<uint4*>(s_q)[i] = reinterpret_cast<const uint4*>(p.mel_q)[i];
  }
  for (int i = kFeMagLive + tid; i < kFeRegionFloats; i += kFeThreads) win[i] = 0.0f;   // bins 201..203 (200 is rewritten)

  const int pair = tid / fft::kR;
  const int col = tid - pair * fft::kR;
  cpx* my_buf = buf + pair * fft::kBufSlots;
  const float* my_win = win + pair * (kFeBlock + kFeSkew) + col;
  const cpx* my_tw = twp + fft::tw_base(warp, lane);
  float* out_tile = reinterpret_cast<float*>(buf);
  const long items = p.S * p.groups;
  // stream of a work item: no division for the server's one-item chunks, a 32-bit one whenever the item count allows
  const bool items32 = items < (1L << 32);
  auto stream_of = [&](long item) -> long {
    if (p.groups == 1) return item;
    if (items32) return static_cast<long>(static_cast<unsigned>(item) / static_cast<unsigned>(p.groups));
    return item / p.groups;
  };
  const bool i16 = p.src.body_dtype == KWS_PCM_I16;
  const int M = p.n_mel;
  const int Mp = M | 1;                               // odd row stride of the [32][M] output tile: conflict-free band writes
  const MelQuad* my_q = (kQuadsInSmem ? s_q : p.mel_q) + warp * p.mel_qpw;
  __syncthreads();                                    // tables staged
  // Barriers per item: window staged | Y' exchanged | Z mirror rows published | magnitudes published | mel tile
  // complete.  The next item's staging writes the window/magnitude region (last read before the fifth barrier) and
  // its stage 1 writes `buf` after its own first barrier, so no barrier is needed at the loop boundary.

  // ---- int16 staging, split in two so that the loads of item i+1 are in flight during the mel projection of item i.
  // Thread t owns the quads of stream samples q0 + 4t + 1280r (r < 5; the fifth round only for t < 60).
  const bool last_quad_ok = tid < kFeLastQuads;
  auto load_quads = [&](long item, int head_len, uint2 (&pre)[kFeQuadRounds]) {
    const long s = stream_of(item);
    const int g = static_cast<int>(item - s * p.groups);
    const int q0 = g * kFeItemHop;
    const int full_len = head_len + p.src.body_len;
    const int total_len = p.total_len<kLens>(s, head_len);       // samples past the length stage as zeros
    // both pointers are indexed by the stream sample number
    const int16_t* body = static_cast<const int16_t*>(p.src.body) + s * p.src.ld_body - head_len;
    const int16_t* head = p.src.head + s * p.src.ld_head;             // only dereferenced below head_len
    if (kLens && g * kFeItemFrames >= frames_of(total_len)) {
      // an item past the stream's last frame loads nothing (the loop below writes its zero rows)
#pragma unroll
      for (int r = 0; r < kFeQuadRounds; ++r) pre[r] = make_uint2(0u, 0u);
      return;
    }
    if (p.vec_ok && ((head_len | full_len) & 3) == 0) {
      // every quad lies entirely in the carried tail, in the chunk, or beyond the signal: one predicated 8-byte load
      // (with lengths, the one quad that straddles a stream's length is masked when it is stored: store_quads)
#pragma unroll
      for (int r = 0; r < kFeQuadRounds; ++r) {
        const int q = q0 + 4 * tid + 4 * kFeThreads * r;
        // the carried tail is shorter than one round (<= 399 samples): only round 0 can read it
        const int16_t* src = (r == 0 && q < head_len ? head : body) + q;
        uint2 v = make_uint2(0u, 0u);
        if (q < total_len && (r < kFeQuadRounds - 1 || last_quad_ok)) v = __ldg(reinterpret_cast<const uint2*>(src));
        pre[r] = v;
      }
    } else {                                                          // odd lengths / unaligned rows: element by element
      auto fetch1 = [&](int q) -> unsigned {
        int x = 0;
        if (q < head_len) x = head[q];
        else if (q < total_len) x = body[q];
        return static_cast<unsigned>(x) & 0xffffu;
      };
#pragma unroll 1
      for (int r = 0; r < kFeQuadRounds; ++r) {
        const int q = q0 + 4 * tid + 4 * kFeThreads * r;
        uint2 v = make_uint2(0u, 0u);
        if (q < total_len && (r < kFeQuadRounds - 1 || last_quad_ok))
          v = make_uint2(fetch1(q) | (fetch1(q + 1) << 16), fetch1(q + 2) | (fetch1(q + 3) << 16));
        // (no dynamic register indexing: the loop is not unrolled)
        if (r == 0) pre[0] = v;
        if (r == 1) pre[1] = v;
        if (r == 2) pre[2] = v;
        if (r == 3) pre[3] = v;
        if (r == 4) pre[4] = v;
      }
    }
  };
  static_assert(kFeQuadRounds == 5, "load_quads' element-wise path names the rounds");
  // window position of sample i is i + 20*(i/320); for i = 4t + 1280r that is 4t + 1360r + 20*(t/80)
  float* my_stage = win + 4 * tid + kFeSkew * (tid / (kFeBlock / 4));
  // returns the thread's sum of |x| over the NEW samples (detector.py:168), exact in fp32 (<= 20 * 32768); samples
  // beyond the signal were loaded as zeros
  auto store_quads = [&](int q0, int head_len, int total_len, const uint2 (&pre)[kFeQuadRounds]) {
    float4 f[kFeQuadRounds];
#pragma unroll
    for (int r = 0; r < kFeQuadRounds; ++r) {
      f[r] = quad_to_float(pre[r]);
      if (kLens) {                                    // the quad that straddles the stream's length: zeros past it
        const int q = q0 + 4 * tid + 4 * kFeThreads * r;
        if (q + 1 >= total_len) f[r].y = 0.0f;
        if (q + 2 >= total_len) f[r].z = 0.0f;
        if (q + 3 >= total_len) f[r].w = 0.0f;
      }
      if (r < kFeQuadRounds - 1 || last_quad_ok) *reinterpret_cast<float4*>(my_stage + (4 * kFeThreads + 4 * kFeSkew) * r) = f[r];
    }
    if (!p.fuse_pre) return 0;
    // sum of |x| over the NEW samples.  The carried tail is shorter than one round (<= 399 samples), so only round 0
    // of the first item can hold old samples; quads beyond the signal were loaded as zeros
    float acc = 0.0f;
#pragma unroll
    for (int r = 1; r < kFeQuadRounds; ++r) acc += (fabsf(f[r].x) + fabsf(f[r].y)) + (fabsf(f[r].z) + fabsf(f[r].w));
    const int q = q0 + 4 * tid;
    acc += (q >= head_len ? fabsf(f[0].x) : 0.0f) + (q + 1 >= head_len ? fabsf(f[0].y) : 0.0f) +
           (q + 2 >= head_len ? fabsf(f[0].z) : 0.0f) + (q + 3 >= head_len ? fabsf(f[0].w) : 0.0f);
    return static_cast<int>(acc);
  };

  long item = blockIdx.x;
  uint2 pre[kFeQuadRounds];
  int head_len = 0;
  if (i16 && item < items) {
    head_len = p.src.head_len ? p.src.head_len[stream_of(item)] : 0;
    load_quads(item, head_len, pre);
  }

  for (; item < items; item += gridDim.x) {
    const long s = stream_of(item);
    const int g = static_cast<int>(item - s * p.groups);
    if (!i16) head_len = p.src.head_len ? p.src.head_len[s] : 0;
    const int total_len = p.total_len<kLens>(s, head_len);
    const int nfr = p.frames(total_len);
    const int q0 = g * kFeItemHop;                    // stream sample held at window position 0
    const int f0 = g * kFeItemFrames;
    // the next item's carried-tail length is needed for its addresses: fetch it a whole item ahead
    const long next = item + gridDim.x;
    int head_len_next = 0;
    if (i16 && next < items && p.src.head_len) head_len_next = p.src.head_len[stream_of(next)];
    if (kLens && p.nframes_out && g == 0 && tid == 0) p.nframes_out[s] = nfr;
    if (kLens && f0 >= nfr) {
      // the item starts past the stream's last frame: zero rows and no PCM (load_quads loaded none), no barrier needed --
      // the next item's staging writes only the window region, whose last reads precede this item
      if (i16 && next < items) load_quads(next, head_len_next, pre);
      p.zero_rows<kFeThreads>(s, f0, f0 + kFeItemFrames, tid);
      head_len = head_len_next;
      continue;
    }

    // ---- stage the window: stream samples [q0, q0 + 5360) -> win[i + 20*(i/320)], zero beyond the signal.
    int vad_acc = 0;
    if (i16) {
      vad_acc = store_quads(q0, head_len, total_len, pre);
    } else {
      // fp32 PCM: thread t takes samples t + 320*r, so the skewed position is simply t + 340*r; samples past the
      // stream's length are zeros (never read)
      const bool last_ok = tid < kFeWinSamples - kFeBlock * (kFeWinRounds - 1);   // the 17th round is partial
      const float* body = static_cast<const float*>(p.src.body) + s * p.src.ld_body + q0 + tid;
#pragma unroll
      for (int r = 0; r < kFeWinRounds; ++r) {
        const int q = q0 + tid + kFeBlock * r;
        const float v = q < total_len ? __ldg(body + kFeBlock * r) : 0.0f;
        if (r < kFeWinRounds - 1 || last_ok) win[tid + (kFeBlock + kFeSkew) * r] = v;
      }
    }
    if (p.fuse_pre) {                                 // block sum of |x| over the chunk (exact integers)
      vad_acc = __reduce_add_sync(0xffffffffu, vad_acc);
      if (lane == 0) red[warp] = vad_acc;
    }
    __syncthreads();

    if (p.fuse_pre) {
      const int keep = tail_keep(total_len);
      const int start = total_len - keep;
      int16_t* tnext = p.pre.tail_next + s * 400;
      if (((start | keep) & 3) == 0 && (reinterpret_cast<uintptr_t>(p.pre.tail_next) & 7) == 0) {
        // whole quads: the first keep/4 (<= 100) threads convert four staged samples back (exact) and store 8 bytes
        if (4 * tid < keep) {
          const int w = start + 4 * tid;
          const float4 f = *reinterpret_cast<const float4*>(win + w + kFeSkew * (w / kFeBlock));
          const unsigned lo = (static_cast<unsigned>(__float2int_rn(f.x)) & 0xffffu) | (static_cast<unsigned>(__float2int_rn(f.y)) << 16);
          const unsigned hi = (static_cast<unsigned>(__float2int_rn(f.z)) & 0xffffu) | (static_cast<unsigned>(__float2int_rn(f.w)) << 16);
          *reinterpret_cast<uint2*>(tnext + 4 * tid) = make_uint2(lo, hi);
        }
      } else {
        for (int i = tid; i < keep; i += kFeThreads) {
          const int w = start + i;
          tnext[i] = static_cast<int16_t>(win[w + kFeSkew * (w / kFeBlock)]);
        }
      }
      if (warp == 0) {                                 // <= 10 partial sums of at most 20 * 32768 each: int is enough
        const int part = lane < kFeWarps ? red[lane] : 0;
        const int sum = __reduce_add_sync(0xffffffffu, part);
        if (lane == 0) p.pre.record(s, sum, nfr, keep, p.nframes_out);
      }
    }

    const int fa = f0 + 2 * pair;
    const bool live = fa < nfr;
    cpx v[20];
    if (live) {
#pragma unroll
      for (int n2 = 0; n2 < 20; ++n2) {
        v[n2].re = my_win[20 * n2 + (n2 >= 16 ? kFeSkew : 0)];
        v[n2].im = my_win[kHop + 20 * n2 + (n2 >= 8 ? kFeSkew : 0)];
      }
      fft::stage1_col(col, v, my_tw, my_buf);
    }
    __syncthreads();
    if (live) fft::stage2_col(col, my_buf, v);
    __syncthreads();
    // magnitudes (times 2, unscaled), transposed (mag_index); the window is dead since the second barrier
    float* mag = win;
    if (live)
      fft::untangle_col(col, v, my_buf, mag + mag_index(col, mag_slot(pair, 0)), mag + mag_index(col, mag_slot(pair, 1)),
                        (fft::kR / 2) * kFeMagStride);
    __syncthreads();
    // ---- the next item's PCM: loads in flight during the mel projection and the output copy
    if (i16 && next < items) load_quads(next, head_len_next, pre);
    // ---- mel projection: lane = frame slot; the warp walks its own flat list of quads (whole bands, dealt out at
    // model creation so that all warps carry the same number of quads).  Weights, row offsets and band ends are
    // warp-uniform broadcast reads; magnitude reads are unit-stride across the lanes; no divergence, no inner loop.
    {
      char* orow = reinterpret_cast<char*>(out_tile + slot_frame(lane) * Mp);
      const char* mcol = reinterpret_cast<const char*>(mag + 2 * lane);
      const float scale = p.mag_scale;
      const MelQuad* rec = my_q;
      float2 acc = make_float2(0.0f, 0.0f);
      auto fetch = [&](const MelQuad* r, float4& w4, int2& me) {
        if (kQuadsInSmem) {
          w4 = *reinterpret_cast<const float4*>(r->w);
          me = *reinterpret_cast<const int2*>(&r->mag_off);
        } else {
          w4 = __ldg(reinterpret_cast<const float4*>(r->w));
          me = __ldg(reinterpret_cast<const int2*>(&r->mag_off));
        }
      };
      auto apply = [&](const float4& w4, const int2& me, const float2& m01, const float2& m23) {
        acc = __ffma2_rn(m01, make_float2(w4.x, w4.y), acc);
        acc = __ffma2_rn(m23, make_float2(w4.z, w4.w), acc);
        if (me.y >= 0) {                                // band complete (predicated, warp-uniform)
          *reinterpret_cast<float*>(orow + me.y) = (acc.x + acc.y) * scale;
          acc = make_float2(0.0f, 0.0f);
        }
      };
#pragma unroll 1
      for (int q = p.mel_qpw; q > 0; q -= 2, rec += 2) {  // two quads per trip, all loads of both issued first
        float4 wa, wb;
        int2 ma, mb;
        fetch(rec, wa, ma);
        fetch(rec + 1, wb, mb);
        const float2 a01 = *reinterpret_cast<const float2*>(mcol + ma.x);
        const float2 a23 = *reinterpret_cast<const float2*>(mcol + ma.x + kFeMagStride * sizeof(float));
        const float2 b01 = *reinterpret_cast<const float2*>(mcol + mb.x);
        const float2 b23 = *reinterpret_cast<const float2*>(mcol + mb.x + kFeMagStride * sizeof(float));
        apply(wa, ma, a01, a23);
        apply(wb, mb, b01, b23);
      }
    }
    __syncthreads();
    // ---- the item's frames are one contiguous block of mel_out
    const int nfi = max(0, min(nfr - f0, kFeItemFrames));
    p.store_tile<kFeThreads>(out_tile, Mp, s, f0, nfi, tid);
    if (kLens) p.zero_rows<kFeThreads>(s, f0 + nfi, f0 + kFeItemFrames, tid);   // the item's frames past the stream's length
    head_len = head_len_next;
  }
}

// Cut the non-zero part of the mel basis [201, M] into quads and deal whole bands to the kFeWarps warps of the
// front-end CTA, longest band first onto the least loaded warp, padding every warp's list to the same length with
// all-zero quads (MelQuad, common.cuh: 4 weights of bins k..k+3 (k even) of one band, the byte offset of
// magnitude row k/2, and the byte offset of the band whose sum is complete after this quad or -1).  Zeros of the basis contribute nothing, so this is exact for any basis.
void build_mel_quads(const float* basis, int M, std::vector<MelQuad>* quads, int* quads_per_warp) {
  struct Band { int b, lo, nq; };
  std::vector<Band> bands;
  for (int b = 0; b < M; ++b) {
    int lo = -1, hi = -1;
    for (int k = 0; k < kBins; ++k)
      if (basis[static_cast<size_t>(k) * M + b] != 0.0f) {
        if (lo < 0) lo = k;
        hi = k;
      }
    if (lo < 0) lo = hi = 0;                               // empty band: one zero quad still writes its 0
    lo &= ~1;                                              // quads start at an even bin (64-bit magnitude reads)
    bands.push_back(Band{b, lo, (hi - lo + 1 + 3) / 4});
  }
  std::stable_sort(bands.begin(), bands.end(), [](const Band& x, const Band& y) { return x.nq > y.nq; });
  std::vector<std::vector<Band>> per_warp(kFeWarps);
  std::vector<int> load(kFeWarps, 0);
  for (const Band& bd : bands) {
    const int w = static_cast<int>(std::min_element(load.begin(), load.end()) - load.begin());
    per_warp[w].push_back(bd);
    load[w] += bd.nq;
  }
  const int qpw = (std::max(1, *std::max_element(load.begin(), load.end())) + 1) & ~1;   // even: two quads per loop trip
  MelQuad zero;
  zero.w[0] = zero.w[1] = zero.w[2] = zero.w[3] = 0.0f;
  zero.mag_off = 0;
  zero.band_off = -1;
  zero.pad[0] = zero.pad[1] = 0;
  quads->assign(static_cast<size_t>(kFeWarps) * qpw, zero);
  for (int w = 0; w < kFeWarps; ++w) {
    size_t at = static_cast<size_t>(w) * qpw;
    for (const Band& bd : per_warp[w])
      for (int j = 0; j < bd.nq; ++j, ++at) {
        MelQuad& q = (*quads)[at];
        for (int e = 0; e < 4; ++e) {
          const int k = bd.lo + 4 * j + e;                 // bins 201..203 of the magnitude array are zero
          q.w[e] = k < kBins ? basis[static_cast<size_t>(k) * M + bd.b] : 0.0f;
        }
        q.mag_off = ((bd.lo + 4 * j) / 2) * kFeMagStride * static_cast<int>(sizeof(float));
        q.band_off = j == bd.nq - 1 ? bd.b * static_cast<int>(sizeof(float)) : -1;
      }
  }
  *quads_per_warp = qpw;
}

static bool quads_in_smem(const kws_model* m) { return kFeWarps * m->mel.quads_per_warp <= kFeQuadSmemMax; }
static size_t frontend_smem_bytes(const kws_model* m) {
  return sizeof(cpx) * fft::kTwSlots + sizeof(cpx) * kFePairs * fft::kBufSlots + sizeof(float) * kFeRegionFloats +
         sizeof(int) * 16 + (quads_in_smem(m) ? sizeof(MelQuad) * kFeWarps * m->mel.quads_per_warp : 0);
}

bool frontend_can_fuse_pre(const kws_model* m, int chunk_len, int tail_cap) {
  // the whole [tail | chunk] must fit one work item: 32 frames / 5360 samples here, 30 frames (<= 5199 samples) on
  // the tensor-core kernel
  if (frontend_uses_tc(m, KWS_PCM_I16)) return chunk_len + tail_cap - 1 <= kFft + kHop * (frontend_tc_item_frames() - 1) + kHop - 1;
  return chunk_len + tail_cap - 1 <= kFeWinSamples;
}

int launch_frontend(const kws_model* m, const PcmSource& src, int64_t S, int32_t max_frames, float* mel_out,
                    cudaStream_t st, const FrontendPre* pre, bool tiled_out, int32_t* nframes_out) {
  if (S <= 0) return KWS_OK;
  if (max_frames <= 0 && !pre) return KWS_OK;
  const bool tc = frontend_uses_tc(m, src.body_dtype);
  FrontendIo io;
  io.src = src;
  io.S = S;
  io.max_frames = max_frames;
  io.groups = static_cast<int>(ceil_div(max_frames > 0 ? max_frames : 1, tc ? frontend_tc_item_frames() : kFeItemFrames));
  io.n_mel = m->cfg.n_mel;
  io.mel_out = mel_out;
  io.tiled_out = tiled_out ? 1 : 0;
  io.tile_chunks = tiled_out ? mel_tile_chunks(m) : 1;
  io.tile_split = tiled_out && mel_tile_split(m) ? 1 : 0;
  io.c_magic = static_cast<unsigned>(((1ull << 32) + io.tile_chunks - 1) / io.tile_chunks);
  io.q_magic = m->cfg.n_mel >= 4 ? static_cast<unsigned>(((1ull << 32) + (m->cfg.n_mel / 4) - 1) / (m->cfg.n_mel / 4)) : 0u;
  io.nframes_out = nframes_out;
  io.fuse_pre = pre ? 1 : 0;
  if (pre) {
    if (io.groups != 1 || src.body_dtype != KWS_PCM_I16 || !nframes_out)
      return fail(KWS_ERR_INVALID_ARGUMENT, "fused pre-step needs an int16 chunk that fits one work item, and nframes_out");
    if (src.lengths) return fail(KWS_ERR_INVALID_ARGUMENT, "the fused pre-step takes no stream lengths");
    io.pre = *pre;
  }
  if (tc) return launch_frontend_tc(m, io, st);

  FrontendParams p{io};
  p.twiddle = reinterpret_cast<const cpx*>(m->twiddle400);
  p.mel_q = m->mel.quads;
  p.mel_qpw = m->mel.quads_per_warp;
  p.vec_ok = (reinterpret_cast<uintptr_t>(src.body) % 8 == 0 && src.ld_body % 4 == 0 &&
              reinterpret_cast<uintptr_t>(src.head) % 8 == 0 && src.ld_head % 4 == 0) ? 1 : 0;
  p.mag_scale = src.body_dtype == KWS_PCM_I16 ? 0.5f / 32768.0f : 0.5f;
  const bool in_smem = quads_in_smem(m), lens = src.lengths != nullptr;
  auto kernel = in_smem ? (lens ? frontend_kernel<true, true> : frontend_kernel<true, false>)
                        : (lens ? frontend_kernel<false, true> : frontend_kernel<false, false>);
  const size_t smem = frontend_smem_bytes(m);
  // the attribute is per device: set it on every launch (a few hundred ns), never cached per thread
  KWS_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  int per_sm = 0;
  KWS_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kFeThreads, smem));
  if (per_sm < 1) return fail(KWS_ERR_CUDA, "frontend_kernel does not fit on an SM (smem %zu)", smem);
  const long items = S * p.groups;
  long blocks = items;
  const long resident = static_cast<long>(per_sm) * sm_count();
  if (blocks > resident) blocks = resident;
  kernel<<<static_cast<unsigned>(blocks), kFeThreads, smem, st>>>(p);
  KWS_LAUNCH_OK("frontend_kernel");
  return KWS_OK;
}

}  // namespace kws

// Debug / test hook (host only, no device needed): the per-warp mel quad lists of a basis [201, M].
// quads_out receives up to `capacity` records of 8 ints {w0,w1,w2,w3 (float bits), magnitude byte offset, band byte
// offset or -1, 0, 0} in warp-major order; returns quads per warp (all 10 warps carry the same number), or a
// negative error code.
extern "C" int kws_debug_mel_quads(const float* basis, int n_mel, int* quads_out, int capacity) {
  kws::clear_error();
  if (!basis || n_mel < 1 || n_mel > kws::kMaxMel) return kws::fail(KWS_ERR_INVALID_ARGUMENT, "bad basis / n_mel");
  std::vector<kws::MelQuad> quads;
  int qpw = 0;
  kws::build_mel_quads(basis, n_mel, &quads, &qpw);
  static_assert(sizeof(kws::MelQuad) == 32, "record layout");
  const int n = static_cast<int>(quads.size());
  if (quads_out) {
    if (capacity < n) return kws::fail(KWS_ERR_INVALID_ARGUMENT, "capacity %d < %d quads", capacity, n);
    memcpy(quads_out, quads.data(), sizeof(kws::MelQuad) * n);
  }
  return qpw;
}

