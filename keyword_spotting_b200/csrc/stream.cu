// Streaming server: the HotwordDetector.start loop (detector.py:148-209) for S lock-step
// streams, every piece of per-stream state resident in HBM.
//
// Per chunk and stream, in the reference's order:
//   1. VAD on the NEW samples: sum|x| > 30 (utils/basic_vad.py:17-18, detector.py:168).
//      Done in exact integer arithmetic on the int16 PCM: sum|x_i16| > 30*32768.
//      Silence -> GRU state zeroed and decision window cleared (detector.py:171-177).
//   2. carried tail ++ chunk; keep (len-400)%160+240 samples for next time (detector.py:179-183)
//   3. model call on the concatenation (detector.py:190-193)         -> K1, K2+K3
//   4. window.add(softmax) with at most 15 chunks (utils/queue.py:16-38, detector.py:195)
//   5. ctc_decode2 over the whole window (detector.py:197-200), ctc_predict(.., '1233')
//   6. trigger -> window cleared, state zeroed (detector.py:201-208)
// The window keeps, per frame, only what ctc_decode2 consumes: the above-threshold winner
// column or -1 (one byte), so re-decoding the 450-frame window every chunk costs 480 B of
// reads per stream instead of 10.8 KB of fp32 probabilities.
#include <atomic>
#include <cstring>
#include <mutex>

#include "common.cuh"
#include "decode_core.cuh"
#include "stream_internal.cuh"

namespace kws {

constexpr int kTailCap = 400;

// One warp per stream: the pre-step of a chunk that the front end cannot take in one work item.
__global__ void __launch_bounds__(256)
stream_pre_kernel(const int16_t* __restrict__ pcm, long ld, int chunk_len, long S, const int16_t* __restrict__ tail_cur,
                  const int* __restrict__ len_cur, const FrontendPre pre, int* __restrict__ nframes, int max_frames) {
  const long s = (blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= S) return;
  const int16_t* row = pcm + s * ld;
  long long sum = 0;
  if (((reinterpret_cast<uintptr_t>(row) & 3) == 0)) {
    const int pairs = chunk_len >> 1;
    const unsigned* row2 = reinterpret_cast<const unsigned*>(row);
    int acc = 0;
    for (int i = lane; i < pairs; i += 32) {
      const unsigned v = __ldg(row2 + i);
      const int a = static_cast<short>(v & 0xffffu), b = static_cast<short>(v >> 16);
      acc += abs(a) + abs(b);            // |int16| <= 32768; a lane sums < 2^31 for chunks < 2^21 samples
    }
    sum = acc;
    if ((chunk_len & 1) && lane == 0) sum += abs(static_cast<int>(row[chunk_len - 1]));
  } else {
    int acc = 0;
    for (int i = lane; i < chunk_len; i += 32) acc += abs(static_cast<int>(row[i]));
    sum = acc;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const int head = len_cur[s];
  const int total = head + chunk_len;
  const int nfr = frames_of(total);
  const int keep = tail_keep(total);
  if (lane == 0) pre.record(s, sum, nfr < max_frames ? nfr : max_frames, keep, nframes);
  const int16_t* tcur = tail_cur + s * kTailCap;
  int16_t* tnext = pre.tail_next + s * kTailCap;
  for (int i = lane; i < keep; i += 32) {
    const int gidx = total - keep + i;
    tnext[i] = gidx < head ? tcur[gidx] : row[gidx - head];
  }
}

struct TokRow {
  const float* p;
  int C;
  __device__ __forceinline__ float operator()(int t, int c) const { return __ldg(p + t * C + 1 + c); }
};

// One thread per stream: push this chunk's tokens, re-decode the window, trigger side effects.
__global__ void __launch_bounds__(128)
stream_post_kernel(const float* __restrict__ probs, int n_step, int C, long S, int W, int fpad,
                   double thres, dec::Keyword kw, const unsigned char* __restrict__ silence,
                   const int* __restrict__ nframes, signed char* __restrict__ tok,
                   unsigned char* __restrict__ slot_frames, int* __restrict__ win_head,
                   int* __restrict__ win_n, float* __restrict__ state, int layers,
                   int* __restrict__ trigger_a, int* __restrict__ trigger_b) {
  const long s = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  if (s >= S) return;
  int head = win_head[s], n = win_n[s];
  if (silence[s]) {            // prob_queue.clear()  (detector.py:177)
    head = 0;
    n = 0;
  }
  // SimpleQueue.add (utils/queue.py:29-35)
  if (n == W) head = (head + 1) % W; else ++n;
  const int slot = (head + n - 1) % W;
  const int nf = nframes[s];
  signed char* trow = tok + (s * W + slot) * static_cast<long>(fpad);
  TokRow row{probs + s * static_cast<long>(n_step) * C, C};
  for (int t = 0; t < nf; ++t) trow[t] = static_cast<signed char>(dec::frame_token(row, t, C - 2, thres));
  slot_frames[s * W + slot] = static_cast<unsigned char>(nf);
  // ctc_decode2 over the concatenated window (detector.py:197-200) + ctc_predict
  dec::Sink sink;
  sink.init(nullptr, 0, kw);
  int prev = -1;
  for (int q = 0; q < n; ++q) {
    const int sl = (head + q) % W;
    const signed char* r = tok + (s * W + sl) * static_cast<long>(fpad);
    const int f = slot_frames[s * W + sl];
    for (int t = 0; t < f; ++t) {
      const int tk = r[t];
      if (tk >= 0) {
        if (prev == -1 || prev != tk) sink.push(tk + 1);
        prev = tk;
      } else {
        prev = -1;
      }
    }
  }
  const int hit = sink.hit;
  if (hit) {                   // detector.py:201-208: clear the window, zero the state
    head = 0;
    n = 0;
    for (int l = 0; l < layers; ++l) {
      float4* h = reinterpret_cast<float4*>(state + (static_cast<long>(l) * S + s) * kHidden);
      for (int i = 0; i < kHidden / 4; ++i) h[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  win_head[s] = head;
  win_n[s] = n;
  if (trigger_a) trigger_a[s] = hit;
  if (trigger_b) trigger_b[s] = hit;
}

__global__ void __launch_bounds__(128)
stream_labels_kernel(long S, int W, int fpad, dec::Keyword kw, const signed char* __restrict__ tok,
                     const unsigned char* __restrict__ slot_frames, const int* __restrict__ win_head,
                     const int* __restrict__ win_n, int* __restrict__ labels, int max_labels,
                     int* __restrict__ counts) {
  const long s = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  if (s >= S) return;
  const int head = win_head[s], n = win_n[s];
  dec::Sink sink;
  sink.init(labels ? labels + s * max_labels : nullptr, max_labels, kw);
  int prev = -1;
  for (int q = 0; q < n; ++q) {
    const int sl = (head + q) % W;
    const signed char* r = tok + (s * W + sl) * static_cast<long>(fpad);
    const int f = slot_frames[s * W + sl];
    for (int t = 0; t < f; ++t) {
      const int tk = r[t];
      if (tk >= 0) {
        if (prev == -1 || prev != tk) sink.push(tk + 1);
        prev = tk;
      } else {
        prev = -1;
      }
    }
  }
  sink.finish();
  if (counts) counts[s] = sink.count();
}

// zero the carried state of silent streams when a chunk produces no frame at all
__global__ void zero_silent_state_kernel(float* state, long S, int layers, const unsigned char* silence) {
  const long idx = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  const long total = static_cast<long>(layers) * S * kHidden;
  if (idx >= total) return;
  const long s = (idx / kHidden) % S;
  if (silence[s]) state[idx] = 0.0f;
}

// ---- per-stream records (layout in include/kws_b200.h).  Every section starts and ends on a 16-byte boundary, so
// both kernels move whole 16-byte pieces: one warp per record, lane-strided over its pieces.
constexpr uint32_t kRecMagic = 0x5253574bu;   // "KWSR" as little-endian bytes
constexpr uint32_t kRecVersion = 1;
constexpr int kRecHeadPieces = 3;             // 48-byte header
constexpr int kRecTailPieces = kTailCap * 2 / 16;

struct RecordGeom {
  long long total;                            // ids in [0, total)
  long long per;                              // streams per object
  int layers, W, fpad, max_frames, max_token;
  int p_tail, p_slots, p_tok, pieces;         // section offsets in pieces (the state starts at kRecHeadPieces)
  __device__ __forceinline__ uint4 head0() const { return make_uint4(kRecMagic, kRecVersion, layers, kHidden); }
  __device__ __forceinline__ uint4 head1() const { return make_uint4(W, fpad, pieces * 16, 0); }
};

static RecordGeom record_geom(const kws_stream* st, long long total) {
  RecordGeom g;
  g.total = total;
  g.per = st->S;
  g.layers = st->model->cfg.num_layers;
  g.W = st->cfg.window_chunks;
  g.fpad = st->fpad;
  g.max_frames = st->max_frames;
  g.max_token = st->model->cfg.num_classes - 3;
  g.p_tail = kRecHeadPieces + g.layers * kHidden / 4;
  g.p_slots = g.p_tail + kRecTailPieces;
  g.p_tok = g.p_slots + (g.W + 15) / 16;
  g.pieces = g.p_tok + g.W * g.fpad / 16;
  return g;
}

// v with bytes [keep, 16) zeroed
__device__ __forceinline__ uint4 keep_bytes(uint4 v, int keep) {
  uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int k = keep - 4 * i;
    w[i] = k >= 4 ? w[i] : k <= 0 ? 0u : w[i] & ((1u << (8 * k)) - 1u);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}

__device__ __forceinline__ bool record_target(const RecordGeom& g, const RecordSlots& one, const RecordSlots* table,
                                              long long id, RecordSlots& o, long& s) {
  if (id < 0 || id >= g.total) return false;
  if (table) {
    o = table[id / g.per];
    s = static_cast<long>(id % g.per);
  } else {
    o = one;
    s = static_cast<long>(id);
  }
  return true;
}

__global__ void __launch_bounds__(256)
stream_export_kernel(const int64_t* __restrict__ ids, long n, const RecordGeom g, const RecordSlots one,
                     const RecordSlots* __restrict__ table, uint4* __restrict__ records) {
  const long r = (blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= n) return;
  uint4* rec = records + r * static_cast<long>(g.pieces);
  const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
  RecordSlots o;
  long s = 0;
  if (!record_target(g, one, table, ids[r], o, s)) {     // all zero: import rejects it (magic 0)
    for (int p = lane; p < g.pieces; p += 32) rec[p] = zero;
    return;
  }
  const int W = g.W, fpad = g.fpad;
  const int tlen = o.tail_len[s], wn = o.win_n[s], wh = o.win_head[s];
  const uint4* state = reinterpret_cast<const uint4*>(o.state + s * kHidden);
  const uint4* tail = reinterpret_cast<const uint4*>(o.tail + s * kTailCap);
  const unsigned char* sf = o.slot_frames + s * W;
  const signed char* tok = o.tok + s * W * static_cast<long>(fpad);
  for (int p = lane; p < g.pieces; p += 32) {
    uint4 v = zero;
    if (p < kRecHeadPieces) {
      v = p == 0 ? g.head0() : p == 1 ? g.head1() : make_uint4(tlen, wn, 0u, 0u);
    } else if (p < g.p_tail) {
      const int q = p - kRecHeadPieces, l = q / (kHidden / 4), i = q % (kHidden / 4);
      v = state[l * g.per * (kHidden / 4) + i];
    } else if (p < g.p_slots) {
      const int j = p - g.p_tail;                          // samples 8j .. 8j+7
      if (8 * j < tlen) v = keep_bytes(tail[j], 2 * (tlen - 8 * j));
    } else if (p < g.p_tok) {
      uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        const int q = 16 * (p - g.p_slots) + k;            // window entry q, oldest first
        if (q < wn) w[k >> 2] |= static_cast<uint32_t>(sf[(wh + q) % W]) << (8 * (k & 3));
      }
      v = make_uint4(w[0], w[1], w[2], w[3]);
    } else {
      const int b = 16 * (p - g.p_tok), q = b / fpad, t0 = b % fpad;
      if (q < wn) {
        const int sl = (wh + q) % W, f = sf[sl];
        if (t0 < f) v = keep_bytes(*reinterpret_cast<const uint4*>(tok + sl * fpad + t0), f - t0);
      }
    }
    rec[p] = v;
  }
}

// Status per record: 0 imported, 1 id out of range, 2 header of another layout, 3 malformed field.  Every field is
// checked before anything is written, so a rejected record leaves its stream untouched.
__global__ void __launch_bounds__(256)
stream_import_kernel(const int64_t* __restrict__ ids, long n, const RecordGeom g, const RecordSlots one,
                     const RecordSlots* __restrict__ table, const uint4* __restrict__ records,
                     int32_t* __restrict__ status) {
  const long r = (blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= n) return;
  const uint4* rec = records + r * static_cast<long>(g.pieces);
  const unsigned char* rsf = reinterpret_cast<const unsigned char*>(rec + g.p_slots);
  const int W = g.W, fpad = g.fpad;
  RecordSlots o;
  long s = 0;
  int st = 0, tlen = 0, wn = 0;
  if (!record_target(g, one, table, ids[r], o, s)) {
    st = 1;
  } else {
    const uint4 h0 = rec[0], h1 = rec[1], h2 = rec[2], e0 = g.head0(), e1 = g.head1();
    tlen = static_cast<int>(h2.x);
    wn = static_cast<int>(h2.y);
    if (h0.x != e0.x || h0.y != e0.y || h0.z != e0.z || h0.w != e0.w || h1.x != e1.x || h1.y != e1.y || h1.z != e1.z) {
      st = 2;
    } else if (tlen < 0 || tlen >= kTailCap || wn < 0 || wn > W) {
      st = 3;
    } else {
      bool bad = false;
      for (int q = lane; q < wn; q += 32) bad |= rsf[q] > g.max_frames;
      for (int p = g.p_tok + lane; p < g.pieces && !bad; p += 32) {
        const int b = 16 * (p - g.p_tok), q = b / fpad, t0 = b % fpad;
        if (q >= wn) break;                                // pieces only grow in q
        const int f = rsf[q];
        if (t0 >= f || f > g.max_frames) continue;
        const uint4 v = rec[p];
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const int tk = static_cast<signed char>(w[k >> 2] >> (8 * (k & 3)));
          bad |= t0 + k < f && (tk < -1 || tk > g.max_token);
        }
      }
      if (__any_sync(0xffffffffu, bad)) st = 3;
    }
  }
  if (lane == 0 && status) status[r] = st;
  if (st != 0) return;
  for (int p = lane; p < g.pieces; p += 32) {
    if (p < kRecHeadPieces) continue;
    if (p < g.p_tail) {
      const int q = p - kRecHeadPieces, l = q / (kHidden / 4), i = q % (kHidden / 4);
      reinterpret_cast<uint4*>(o.state + (static_cast<long>(l) * g.per + s) * kHidden)[i] = rec[p];
    } else if (p < g.p_slots) {
      const int j = p - g.p_tail;
      reinterpret_cast<uint4*>(o.tail + s * kTailCap)[j] = keep_bytes(rec[p], 2 * (tlen - 8 * j));
    } else if (p < g.p_tok) {
      for (int k = 0; k < 16; ++k) {
        const int q = 16 * (p - g.p_slots) + k;
        if (q < W) o.slot_frames[s * W + q] = q < wn ? rsf[q] : 0;
      }
    } else {
      const int b = 16 * (p - g.p_tok), q = b / fpad, t0 = b % fpad;
      const int keep = q < wn ? rsf[q] - t0 : 0;
      *reinterpret_cast<uint4*>(o.tok + (s * W + q) * static_cast<long>(fpad) + t0) = keep_bytes(rec[p], keep);
    }
  }
  if (lane == 0) {
    o.tail_len[s] = tlen;
    o.win_head[s] = 0;
    o.win_n[s] = wn;
  }
}

template <typename T>
static int dev_alloc(T** p, size_t n, bool zero) {
  *p = nullptr;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(p), sizeof(T) * (n ? n : 1));
  if (e != cudaSuccess) return fail(KWS_ERR_ALLOC, "cudaMalloc(%zu) failed: %s", sizeof(T) * n, cudaGetErrorString(e));
  if (zero) KWS_CUDA_OK(cudaMemset(*p, 0, sizeof(T) * (n ? n : 1)));
  return KWS_OK;
}

static void free_stream(kws_stream* st) {
  if (!st) return;
  cudaFree(st->state);
  for (int i = 0; i < 2; ++i) {
    cudaFree(st->tail[i]);
    cudaFree(st->tail_len[i]);
    cudaFree(st->pcm_dev[i]);
    if (st->copied[i]) cudaEventDestroy(st->copied[i]);
    if (st->consumed[i]) cudaEventDestroy(st->consumed[i]);
  }
  if (st->copy_stream) cudaStreamDestroy(st->copy_stream);
  cudaFree(st->silence);
  cudaFree(st->nframes);
  cudaFree(st->mel);
  cudaFree(st->seq);
  cudaFree(st->y_rows);
  cudaFree(st->probs);
  cudaFree(st->tok);
  cudaFree(st->slot_frames);
  cudaFree(st->win_head);
  cudaFree(st->win_n);
  cudaFree(st->trigger);
  delete st;
}

static int frames_for_chunk(int chunk_len) { return frames_of(chunk_len + kTailCap - 1); }   // with the longest tail (399)

RecordSlots record_slots(const kws_stream* st) {
  RecordSlots o;
  o.state = st->state;
  o.tail = st->tail[st->cur];
  o.tail_len = st->tail_len[st->cur];
  o.tok = st->tok;
  o.slot_frames = st->slot_frames;
  o.win_head = st->win_head;
  o.win_n = st->win_n;
  return o;
}

int64_t record_bytes(const kws_stream* st) { return 16LL * record_geom(st, 0).pieces; }

static int check_record_args(const kws_stream* st, const int64_t* ids, int64_t n, const void* records) {
  KWS_REQUIRE(st != nullptr, "stream handle is NULL");
  KWS_REQUIRE(n >= 0, "n must be >= 0");
  KWS_REQUIRE(n == 0 || (ids != nullptr && records != nullptr), "ids / records are NULL");
  KWS_REQUIRE(reinterpret_cast<uintptr_t>(records) % 16 == 0, "records must be 16-byte aligned");
  return KWS_OK;
}

int launch_record_export(const kws_stream* st, const RecordSlots* table, int64_t total, const int64_t* ids, int64_t n,
                         void* records, cudaStream_t cs) {
  const int rc = check_record_args(st, ids, n, records);
  if (rc != KWS_OK || n == 0) return rc;
  stream_export_kernel<<<static_cast<unsigned>(ceil_div(n * 32, 256)), 256, 0, cs>>>(
      ids, n, record_geom(st, total), record_slots(st), table, static_cast<uint4*>(records));
  KWS_LAUNCH_OK("stream_export_kernel");
  return KWS_OK;
}

int launch_record_import(const kws_stream* st, const RecordSlots* table, int64_t total, const int64_t* ids, int64_t n,
                         const void* records, int32_t* status_out, cudaStream_t cs) {
  const int rc = check_record_args(st, ids, n, records);
  if (rc != KWS_OK || n == 0) return rc;
  stream_import_kernel<<<static_cast<unsigned>(ceil_div(n * 32, 256)), 256, 0, cs>>>(
      ids, n, record_geom(st, total), record_slots(st), table, static_cast<const uint4*>(records), status_out);
  KWS_LAUNCH_OK("stream_import_kernel");
  return KWS_OK;
}

}  // namespace kws

using namespace kws;

extern "C" int kws_stream_create(kws_model* m, const kws_stream_config* cfg, kws_stream** out) {
  clear_error();
  KWS_REQUIRE(m && cfg && out, "NULL argument");
  *out = nullptr;
  KWS_REQUIRE(cfg->n_streams >= 1, "n_streams must be >= 1");
  KWS_REQUIRE(cfg->max_chunk >= 1 && cfg->max_chunk <= (1 << 20), "max_chunk out of range");
  KWS_REQUIRE(cfg->window_chunks >= 1 && cfg->window_chunks <= 255, "window_chunks must be in [1, 255]");
  KWS_REQUIRE(cfg->vad_threshold >= 0, "vad_threshold must be >= 0");
  KWS_REQUIRE(m->cfg.num_classes >= 3 && m->cfg.num_classes <= 11, "streaming decode needs 3..11 classes");
  KWS_REQUIRE(std::memchr(cfg->keyword, 0, sizeof(cfg->keyword)) != nullptr && std::strlen(cfg->keyword) <= 16,
              "keyword must be a NUL-terminated string of at most 16 characters");
  const int mf = frames_for_chunk(cfg->max_chunk);
  KWS_REQUIRE(mf <= 255, "max_chunk produces more than 255 frames per chunk");
  KWS_CUDA_OK(cudaSetDevice(m->device));
  kws_stream* st = new kws_stream();
  st->model = m;
  st->device = m->device;
  st->cfg = *cfg;
  st->S = cfg->n_streams;
  st->max_frames = mf;
  st->fpad = (mf + 15) / 16 * 16;
  if (st->fpad == 0) st->fpad = 16;
  st->kw = dec::parse_keyword(cfg->keyword);
  const size_t S = static_cast<size_t>(st->S);
  const int L = m->cfg.num_layers, C = m->cfg.num_classes, M = m->cfg.n_mel, W = cfg->window_chunks;
  int rc = dev_alloc(&st->state, S * L * kHidden, true);
  for (int i = 0; i < 2 && rc == KWS_OK; ++i) {
    rc = dev_alloc(&st->tail[i], S * kTailCap, true);
    if (rc == KWS_OK) rc = dev_alloc(&st->tail_len[i], S, true);
  }
  if (rc == KWS_OK) rc = dev_alloc(&st->silence, S, true);
  if (rc == KWS_OK) rc = dev_alloc(&st->nframes, S, true);
  if (rc == KWS_OK) rc = dev_alloc(&st->mel, mel_scratch_elems(st->S, mf, M), false);
  if (rc == KWS_OK) rc = dev_alloc(&st->probs, S * (mf ? mf : 1) * C, false);
  if (rc == KWS_OK) rc = dev_alloc(&st->tok, S * W * st->fpad, true);
  if (rc == KWS_OK) rc = dev_alloc(&st->slot_frames, S * W, true);
  if (rc == KWS_OK) rc = dev_alloc(&st->win_head, S, true);
  if (rc == KWS_OK) rc = dev_alloc(&st->win_n, S, true);
  if (rc == KWS_OK) rc = dev_alloc(&st->trigger, S, true);
  if (rc == KWS_OK && mf > 0 && L > 1) rc = dev_alloc(&st->seq, seq_scratch_elems(st->S, mf, L), false);
  if (rc == KWS_OK && mf > 0 && m->octbit) rc = dev_alloc(&st->y_rows, S * mf * kHidden, false);
  if (rc != KWS_OK) {
    free_stream(st);
    return rc;
  }
  *out = st;
  return KWS_OK;
}

extern "C" int kws_stream_destroy(kws_stream* st) {
  clear_error();
  if (st) {
    cudaSetDevice(st->device);
    cudaDeviceSynchronize();
    free_stream(st);
  }
  return KWS_OK;
}

extern "C" int kws_stream_reset(kws_stream* st, void* stream) {
  clear_error();
  KWS_REQUIRE(st != nullptr, "stream handle is NULL");
  cudaStream_t cs = static_cast<cudaStream_t>(stream);
  const size_t S = static_cast<size_t>(st->S);
  KWS_CUDA_OK(cudaSetDevice(st->model->device));
  KWS_CUDA_OK(cudaMemsetAsync(st->state, 0, sizeof(float) * S * st->model->cfg.num_layers * kHidden, cs));
  for (int i = 0; i < 2; ++i) KWS_CUDA_OK(cudaMemsetAsync(st->tail_len[i], 0, sizeof(int32_t) * S, cs));
  KWS_CUDA_OK(cudaMemsetAsync(st->win_head, 0, sizeof(int32_t) * S, cs));
  KWS_CUDA_OK(cudaMemsetAsync(st->win_n, 0, sizeof(int32_t) * S, cs));
  return KWS_OK;
}

extern "C" int32_t kws_stream_max_frames(const kws_stream* st) { return st ? st->max_frames : 0; }
extern "C" const float* kws_stream_state(const kws_stream* st) { return st ? st->state : nullptr; }

extern "C" int kws_stream_copy_state(kws_stream* st, float* state_out, void* stream) {
  clear_error();
  KWS_REQUIRE(st != nullptr && state_out != nullptr, "NULL argument");
  KWS_CUDA_OK(cudaSetDevice(st->model->device));
  KWS_CUDA_OK(cudaMemcpyAsync(state_out, st->state,
                              sizeof(float) * st->S * st->model->cfg.num_layers * kHidden,
                              cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  return KWS_OK;
}

extern "C" int64_t kws_stream_record_bytes(const kws_stream* st) { return st ? record_bytes(st) : 0; }

extern "C" int kws_stream_export(kws_stream* st, const int64_t* ids, int64_t n, void* records, void* stream) {
  clear_error();
  KWS_REQUIRE(st != nullptr, "stream handle is NULL");
  KWS_CUDA_OK(cudaSetDevice(st->device));
  return launch_record_export(st, nullptr, st->S, ids, n, records, static_cast<cudaStream_t>(stream));
}

extern "C" int kws_stream_import(kws_stream* st, const int64_t* ids, int64_t n, const void* records,
                                 int32_t* status_out, void* stream) {
  clear_error();
  KWS_REQUIRE(st != nullptr, "stream handle is NULL");
  KWS_CUDA_OK(cudaSetDevice(st->device));
  return launch_record_import(st, nullptr, st->S, ids, n, records, status_out, static_cast<cudaStream_t>(stream));
}

// Debug: device time of the three parts of a step (front end incl. the fused pre-step | GRU layers | decode + trigger),
// measured with CUDA events on the step's stream.  Enabling it makes every step synchronise -- never on in production.
static std::atomic<int> g_step_timing_on{0};
static std::mutex g_step_mutex;                    // the sums may be fed by stream objects on several host threads
static double g_step_ms[3] = {0.0, 0.0, 0.0};
static long g_step_count = 0;
extern "C" int kws_debug_step_timing(int enable, double* ms_out3, long long* steps_out) {
  kws::clear_error();
  std::lock_guard<std::mutex> lock(g_step_mutex);
  if (ms_out3) {
    for (int i = 0; i < 3; ++i) ms_out3[i] = g_step_ms[i];
  }
  if (steps_out) *steps_out = g_step_count;
  if (enable != g_step_timing_on) {
    g_step_timing_on = enable;
    g_step_ms[0] = g_step_ms[1] = g_step_ms[2] = 0.0;
    g_step_count = 0;
  }
  return KWS_OK;
}

extern "C" int kws_stream_step(kws_stream* st, const int16_t* pcm, int32_t chunk_len, int64_t ld_pcm,
                               int32_t* trigger_out, float* probs_out, int32_t* nframes_out, void* stream) {
  clear_error();
  KWS_REQUIRE(st != nullptr, "stream handle is NULL");
  KWS_REQUIRE(chunk_len >= 1 && chunk_len <= st->cfg.max_chunk, "chunk_len %d outside [1, max_chunk=%d]", chunk_len,
              st->cfg.max_chunk);
  KWS_REQUIRE(pcm != nullptr, "pcm is NULL");
  KWS_REQUIRE(ld_pcm >= chunk_len, "ld_pcm < chunk_len");
  kws_model* m = st->model;
  cudaStream_t cs = static_cast<cudaStream_t>(stream);
  KWS_CUDA_OK(cudaSetDevice(m->device));
  const long S = st->S;
  const int cur = st->cur, nxt = cur ^ 1;
  const int n_step = frames_for_chunk(chunk_len);
  const int C = m->cfg.num_classes;

  PcmSource src;
  src.body = pcm;
  src.ld_body = ld_pcm;
  src.body_len = chunk_len;
  src.body_dtype = KWS_PCM_I16;
  src.head = st->tail[cur];
  src.ld_head = kTailCap;
  src.head_len = st->tail_len[cur];
  const bool fused = frontend_can_fuse_pre(m, chunk_len, kTailCap);
  const bool tiled = mel_can_tile(m);
  cudaEvent_t tev[4] = {nullptr, nullptr, nullptr, nullptr};
  if (g_step_timing_on) {
    for (int i = 0; i < 4; ++i) KWS_CUDA_OK(cudaEventCreate(&tev[i]));
    KWS_CUDA_OK(cudaEventRecord(tev[0], cs));
  }
  FrontendPre pre;
  pre.vad_limit = static_cast<long long>(st->cfg.vad_threshold) * 32768LL;
  pre.tail_next = st->tail[nxt];
  pre.len_next = st->tail_len[nxt];
  pre.silence = st->silence;
  if (fused) {
    // one pass over the chunk: VAD + tail carry + frame count + framing/FFT/mel
    int rc = launch_frontend(m, src, S, n_step, st->mel, cs, &pre, tiled, st->nframes);
    if (rc != KWS_OK) return rc;
  } else {
    stream_pre_kernel<<<static_cast<unsigned>(ceil_div(S * 32, 256)), 256, 0, cs>>>(
        pcm, ld_pcm, chunk_len, S, st->tail[cur], st->tail_len[cur], pre, st->nframes, n_step);
    KWS_LAUNCH_OK("stream_pre_kernel");
  }

  if (n_step > 0) {
    if (!fused) {
      int rc = launch_frontend(m, src, S, n_step, st->mel, cs, nullptr, tiled);
      if (rc != KWS_OK) return rc;
    }
    if (tev[1]) KWS_CUDA_OK(cudaEventRecord(tev[1], cs));
    int rc = KWS_OK;
    GruArgs a;
    a.x = st->mel;
    a.x_tiled = tiled;
    a.seq_scratch = st->seq;
    a.y_rows_scratch = st->y_rows;
    a.S = S;
    a.n = n_step;
    a.seq_len = st->nframes;
    a.zero_state = st->silence;
    a.state_in = st->state;
    a.state_out = st->state;
    a.probs = st->probs;
    a.logits = nullptr;
    rc = launch_gru(m, a, cs);
    if (rc != KWS_OK) return rc;
  } else {
    const long total = static_cast<long>(m->cfg.num_layers) * S * kHidden;
    zero_silent_state_kernel<<<static_cast<unsigned>(ceil_div(total, 256)), 256, 0, cs>>>(
        st->state, S, m->cfg.num_layers, st->silence);
    KWS_LAUNCH_OK("zero_silent_state_kernel");
  }
  if (tev[2]) KWS_CUDA_OK(cudaEventRecord(tev[2], cs));
  stream_post_kernel<<<static_cast<unsigned>(ceil_div(S, 128)), 128, 0, cs>>>(
      st->probs, n_step, C, S, st->cfg.window_chunks, st->fpad, st->cfg.decode_thres, st->kw, st->silence,
      st->nframes, st->tok, st->slot_frames, st->win_head, st->win_n, st->state, m->cfg.num_layers,
      st->trigger, trigger_out);
  KWS_LAUNCH_OK("stream_post_kernel");
  if (tev[0]) {
    KWS_CUDA_OK(cudaEventRecord(tev[3], cs));
    KWS_CUDA_OK(cudaEventSynchronize(tev[3]));
    if (n_step > 0) {
      std::lock_guard<std::mutex> lock(g_step_mutex);
      for (int i = 0; i < 3; ++i) {
        float ms = 0.0f;
        KWS_CUDA_OK(cudaEventElapsedTime(&ms, tev[i], tev[i + 1]));
        g_step_ms[i] += ms;
      }
      ++g_step_count;
    }
    for (int i = 0; i < 4; ++i) cudaEventDestroy(tev[i]);
  }
  st->cur = nxt;
  if (probs_out && n_step > 0) {
    KWS_CUDA_OK(cudaMemcpy2DAsync(probs_out, sizeof(float) * st->max_frames * C, st->probs,
                                  sizeof(float) * n_step * C, sizeof(float) * n_step * C, S,
                                  cudaMemcpyDeviceToDevice, cs));
  }
  if (nframes_out)
    KWS_CUDA_OK(cudaMemcpyAsync(nframes_out, st->nframes, sizeof(int32_t) * S, cudaMemcpyDeviceToDevice, cs));
  return KWS_OK;
}

extern "C" int kws_stream_step_host(kws_stream* st, const int16_t* pcm_host, int32_t chunk_len,
                                    int32_t* trigger_host, void* stream) {
  clear_error();
  KWS_REQUIRE(st != nullptr, "stream handle is NULL");
  KWS_REQUIRE(chunk_len >= 1 && chunk_len <= st->cfg.max_chunk, "chunk_len %d outside [1, max_chunk=%d]", chunk_len,
              st->cfg.max_chunk);
  KWS_REQUIRE(pcm_host != nullptr, "pcm_host is NULL");
  cudaStream_t cs = static_cast<cudaStream_t>(stream);
  KWS_CUDA_OK(cudaSetDevice(st->model->device));
  const size_t S = static_cast<size_t>(st->S);
  if (!st->copy_stream) {
    KWS_CUDA_OK(cudaStreamCreateWithFlags(&st->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      int rc = dev_alloc(&st->pcm_dev[i], S * st->cfg.max_chunk, false);
      if (rc != KWS_OK) return rc;
      KWS_CUDA_OK(cudaEventCreateWithFlags(&st->copied[i], cudaEventDisableTiming));
      KWS_CUDA_OK(cudaEventCreateWithFlags(&st->consumed[i], cudaEventDisableTiming));
    }
  }
  const int b = st->host_buf;
  // the staging buffer may be overwritten only after the step that read it has finished
  if (st->consumed_valid[b]) KWS_CUDA_OK(cudaStreamWaitEvent(st->copy_stream, st->consumed[b], 0));
  KWS_CUDA_OK(cudaMemcpyAsync(st->pcm_dev[b], pcm_host, sizeof(int16_t) * S * chunk_len, cudaMemcpyHostToDevice,
                              st->copy_stream));
  KWS_CUDA_OK(cudaEventRecord(st->copied[b], st->copy_stream));
  KWS_CUDA_OK(cudaStreamWaitEvent(cs, st->copied[b], 0));
  int rc = kws_stream_step(st, st->pcm_dev[b], chunk_len, chunk_len, nullptr, nullptr, nullptr, stream);
  if (rc != KWS_OK) return rc;
  KWS_CUDA_OK(cudaEventRecord(st->consumed[b], cs));
  st->consumed_valid[b] = true;
  st->host_buf = b ^ 1;
  if (trigger_host)
    KWS_CUDA_OK(cudaMemcpyAsync(trigger_host, st->trigger, sizeof(int32_t) * S, cudaMemcpyDeviceToHost, cs));
  return KWS_OK;
}

extern "C" int kws_stream_labels(kws_stream* st, int32_t* labels_out, int32_t max_labels, int32_t* counts_out,
                                 void* stream) {
  clear_error();
  KWS_REQUIRE(st != nullptr, "stream handle is NULL");
  KWS_REQUIRE(labels_out == nullptr || max_labels >= 1, "max_labels must be >= 1");
  KWS_CUDA_OK(cudaSetDevice(st->model->device));
  stream_labels_kernel<<<static_cast<unsigned>(ceil_div(st->S, 128)), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      st->S, st->cfg.window_chunks, st->fpad, st->kw, st->tok, st->slot_frames, st->win_head, st->win_n,
      labels_out, max_labels, counts_out);
  KWS_LAUNCH_OK("stream_labels_kernel");
  return KWS_OK;
}
