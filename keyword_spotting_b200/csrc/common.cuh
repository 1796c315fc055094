// Shared internals of libkws_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdarg>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/kws_b200.h"

namespace kws {

constexpr int kHidden = 128;      // config/rnn_config.py:84 -- the kernels are built for H = 128
constexpr int kMaxLayers = 4;
constexpr int kMaxClasses = 16;
constexpr int kFft = 400;         // config/rnn_config.py:57
constexpr int kHop = 160;         // config/rnn_config.py:58
constexpr int kBins = kFft / 2 + 1;
constexpr int kMaxMel = 128;

// -------------------------------------------------------------------- errors
void set_error(const char* fmt, ...);
void clear_error();
int fail(int code, const char* fmt, ...);

#define KWS_CUDA_OK(expr)                                                                   \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess)                                                                  \
      return ::kws::fail(KWS_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                         __FILE__, __LINE__);                                               \
  } while (0)

#define KWS_LAUNCH_OK(what)                                                                 \
  do {                                                                                      \
    cudaError_t _e = cudaGetLastError();                                                    \
    if (_e != cudaSuccess)                                                                  \
      return ::kws::fail(KWS_ERR_CUDA, "launch of %s failed: %s", what, cudaGetErrorString(_e)); \
  } while (0)

#define KWS_REQUIRE(cond, ...)                                          \
  do {                                                                  \
    if (!(cond)) return ::kws::fail(KWS_ERR_INVALID_ARGUMENT, __VA_ARGS__); \
  } while (0)

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// -------------------------------------------------------------------- attention_ctc: per-utterance lengths
// T' of T mel frames (models/attention_ctc.py:88-90): kws_attention_frames and every attention kernel use this one rule.
__host__ __device__ __forceinline__ int att_frames(int T, int combine) { return combine > 1 ? T / combine + 1 : T; }

constexpr int kAttCoreTcMaxKeys = 400;   // the tensor-core attention core takes T' <= 400 (attention_tc.cu)

// The lengths of a variable-length attention batch as every kernel sees them: utterance b has lens[b] valid frames,
// clamped to [1, T], and T'_b = att_frames(lens[b], combine) rows.  lens == nullptr: every utterance has T frames.
// The forward pass passes mel frames (T, combine of the model); the single-kernel debug entry points pass rows
// (T = T', combine = 1).  Row strides stay T' = att_frames(T, combine) whatever the lengths.
struct AttLens {
  const int32_t* lens;
  int T;
  int combine;
  __device__ __forceinline__ int frames_in(long b) const { return lens ? min(max(__ldg(lens + b), 1), T) : T; }
  __device__ __forceinline__ int rows_of(long b) const { return att_frames(frames_in(b), combine); }
  // does [r0, r0 + tile) of a [B * Tp, .] activation hold a row of some utterance's first T'_b rows?  (O(1): a tile that
  // reaches the next utterance holds that utterance's row 0, which every utterance has)
  __device__ __forceinline__ bool tile_live(int Tp, long rows, long r0, int tile) const {
    if (!lens) return true;
    const long b0 = r0 / Tp;
    const long rlast = (r0 + tile < rows ? r0 + tile : rows) - 1;
    return r0 - b0 * Tp < rows_of(b0) || (b0 + 1) * Tp <= rlast;
  }
};

int sm_count();   // SMs of the current device (cached)

// -------------------------------------------------------------------- model
struct LayerWeights {
  int in_dim = 0;               // n_mel for layer 0, H above
  float* gates_kernel = nullptr;  // [in+H, 2H] row-major (TF layout)
  float* gates_bias = nullptr;    // [2H]
  float* cand_kernel = nullptr;   // [in+H, H]
  float* cand_bias = nullptr;     // [H]
  // tensor-core path (gru_tc.cu): fp16 B operand [384, tc_kx+H] in the canonical smem layout, fused bias [384]
  int tc_kx = 0;                // x width padded to 16
  int tc_kxw = 0;               // x columns in tc_wpack (2*tc_kx for layer 0: hi and lo parts)
  void* tc_wpack = nullptr;
  float* tc_bias = nullptr;
};

struct OctbitMatrix {           // one OctbitMatMul's constants on the device (gru_octbit.cu)
  signed char* wq = nullptr;    // [B, K] int8, already transposed (octbit_graph.py:191-215)
  float* obias = nullptr;       // [B] the op's bias attr
  float scale = 0.0f;           // the op's scale attr
  int* cand_count = nullptr;    // [B] pairs of the row that can saturate int16
  unsigned short* cand = nullptr;   // [B, K/2]
  int B = 0, K = 0;
};

struct alignas(16) MelQuad {     // 4 consecutive bins (from an even bin) of one mel band
  float w[4];
  int mag_off;                   // byte offset of the bin pair's row in the front end's transposed magnitude array
  int band_off;                  // byte offset of the band in the output row if this quad completes it, else -1
  int pad[2];
};
struct MelSparse {               // non-zero part of the mel basis as per-warp lists of quads (frontend.cu)
  MelQuad* quads = nullptr;      // [10 warps][quads_per_warp]
  int quads_per_warp = 0;
};

struct FrontendDftTables {       // general front end (frontend_dft.cu): every frame other than 400/160
  void* tw = nullptr;            // fp16 twiddles [chunks][hi | lo][ncols x 32], canonical K-major
  void* mel_seg = nullptr;       // int4 [n_mel]: {first bin, bins, offset into mel_w, 0}
  float* mel_w = nullptr;        // the bands' non-zero spans, concatenated
};

struct FrontendTcTables {        // tensor-core front end (frontend_tc.cu)
  bool ready = false;
  uint32_t* tw = nullptr;        // twiddles as TMEM rows [2 tiles][2 parts][128][40]
  void* mel_seg = nullptr;       // int4 [n_mel]: {first bin, bins, offset into mel_w, 0}
  float* mel_w = nullptr;        // the bands' non-zero spans, concatenated, zero-padded to multiples of 8 bins
  int mel_nw = 0;
};

}  // namespace kws

struct kws_model {
  kws_model_config cfg;
  int device = 0;
  int precision = KWS_PRECISION_TC_FP16;
  int frontend = KWS_FRONTEND_FFT;   // K1 formulation (kws_model_set_frontend)
  float* mel_basis = nullptr;     // [fft/2+1, M] dense, as given
  // 400/160 models: the FFT and tensor-core front ends' tables; every other frame: the DFT front end's (fe_dft.tw set)
  kws::MelSparse mel;
  kws::FrontendTcTables fe_tc;
  float2* twiddle400 = nullptr;   // [20*52] periodic k2-major twiddles (fft400.cuh kTwStride)
  kws::FrontendDftTables fe_dft;
  kws::LayerWeights layer[kws::kMaxLayers];
  float* fc_w = nullptr;          // [H, C]
  float* fc_b = nullptr;          // [C]
  std::vector<float> fc_w_host, fc_b_host;   // host copies (the tensor-core kernel takes them as kernel parameters)
  // scratch owned by the model (grown by kws_model_reserve)
  int64_t cap_streams = 0;
  int32_t cap_frames = 0;
  float* scratch_mel = nullptr;   // [S, n, M]
  float* scratch_seq = nullptr;   // layer hand-off [tiles, n, H, 64]
  int32_t* scratch_nfr = nullptr; // [S] frames per stream of a forward over streams of their own lengths
  // the octbit-rewritten graph (kws_model_set_octbit): per layer gates / candidate, and the FC
  bool octbit = false;
  kws::OctbitMatrix oct_gates[kws::kMaxLayers], oct_cand[kws::kMaxLayers], oct_fc;
  float* oct_y_rows = nullptr;    // [S, n, H] last-layer outputs for the FC (non-stream forwards)
  size_t oct_y_cap = 0;
  bool tc_fits = true;            // every layer fits the tensor-core recurrent kernel's shared memory (set at creation)
  void* tc_xt = nullptr;          // row-tiled fp16 copy of a caller's row-major x (kws_gru_forward on the tensor-core path)
  size_t tc_xt_bytes = 0;
  cudaStream_t aux_stream = nullptr;          // second stream + events of the layer pipeline for small batches (gru_tc.cu)
  std::vector<cudaEvent_t> aux_events;
};

namespace kws {

// ---- kernels' host launchers (one per .cu file)
struct PcmSource {
  // sample i of stream s:  i < head_len(s) ? head[s*ld_head + i] : body[s*ld_body + i - head_len(s)]
  const void* body = nullptr;
  int64_t ld_body = 0;
  int32_t body_len = 0;
  int body_dtype = KWS_PCM_F32;
  const int16_t* head = nullptr;      // carried tail (server only), int16
  int64_t ld_head = 0;
  const int32_t* head_len = nullptr;  // [S] or null (= 0)
  // [S] or null (= body_len): valid body samples per stream, clamped to [0, body_len].  Samples at or past it are never
  // read and stage as zeros, so a stream of a padded batch is transformed exactly as the stream alone.
  const int32_t* lengths = nullptr;
  __device__ __forceinline__ int body_valid(long s) const {
    return lengths ? min(max(__ldg(lengths + s), 0), body_len) : body_len;
  }
};

// Chunk rules of the front end and the streaming server.  Frames of a signal of `total` samples (utils/stft.py:60-61),
// 0 below one frame:
__host__ __device__ __forceinline__ int frames_of(int total, int fft, int hop) {
  return total >= fft ? 1 + (total - fft) / hop : 0;
}
// samples carried into the next chunk (detector.py:181-182): the last (total - fft) % hop + fft - hop, or all of them
// while no frame fits
__host__ __device__ __forceinline__ int tail_keep(int total, int fft, int hop) {
  return total >= fft ? (total - fft) % hop + (fft - hop) : total;
}
// the same at 400/160, the frame of the FFT and tensor-core front ends
__host__ __device__ __forceinline__ int frames_of(int total) { return frames_of(total, kFft, kHop); }
__host__ __device__ __forceinline__ int tail_keep(int total) { return tail_keep(total, kFft, kHop); }
// Longest carried tail of a frame of fft samples is fft - 1; its buffer holds max(400, ceil8(fft)) samples per stream
// (400 keeps the record layout of every fft_size <= 400, 16-byte pieces keep the record kernels' moves whole).
inline int tail_capacity(int fft) { return fft <= 400 ? 400 : (fft + 7) / 8 * 8; }

// The streaming server's per-chunk pre-step: VAD flag, frame count and next carried tail.  Fused into the front end
// when the chunk fits one work item (frontend_can_fuse_pre), so that the CTA that stages the chunk produces them and
// the PCM is read once; stream_pre_kernel (stream.cu) otherwise.
struct FrontendPre {
  long long vad_limit = 0;            // speech iff sum|x_i16| > vad_limit
  int16_t* tail_next = nullptr;       // [S, tail capacity] (400 whenever the pre-step is fused)
  int32_t* len_next = nullptr;        // [S]
  unsigned char* silence = nullptr;   // [S]
  // stream s's record, from the sum of |x_i16| over its new samples; its frame count goes to nframes[s]
  __device__ __forceinline__ void record(long s, long long vad_sum, int frames, int keep, int32_t* nframes) const {
    silence[s] = vad_sum > vad_limit ? 0 : 1;
    nframes[s] = frames;
    len_next[s] = keep;
  }
};
bool frontend_can_fuse_pre(const kws_model* m, int chunk_len, int tail_cap);
int build_frontend_tc_tables(kws_model* m, const float* basis /*[201, M] host*/);
void free_frontend_tc_tables(kws_model* m);
// 400/160 runs the FFT / tensor-core front ends; every other frame runs the DFT front end (frontend_dft.cu)
inline bool frontend_is_default_frame(const kws_model* m) { return m->cfg.fft_size == kFft && m->cfg.hop_size == kHop; }
int build_frontend_dft_tables(kws_model* m, const float* basis /*[fft/2+1, M] host*/);
void free_frontend_dft_tables(kws_model* m);
bool frontend_uses_tc(const kws_model* m, int pcm_dtype);
int default_frontend();           // KWS_FRONTEND=tc|fft in the environment, else fft
int frontend_tc_item_frames();
void build_mel_quads(const float* basis /*[201, M] host*/, int M, std::vector<MelQuad>* quads, int* quads_per_warp);
// Stream-tiled mel scratch (front end -> tensor-core GRU, tc05.cuh "row-tiled A operand"): the fp16 MMA operand of
// layer 0, [S/128 tiles][n frames][x_hi chunks | x_lo chunks][128 streams][8 mels]; chunk c holds mels 8c..8c+7 (zero
// past n_mel, up to kx = ceil16(n_mel)), x = x_hi + x_lo.  The front end writes 16-byte pieces that are contiguous
// across streams, the recurrent kernel takes a whole tile-step (kxw/8 * 2048 bytes) with one bulk copy.
// Size: ceil(S/128)*128 * n * 2*kx halves = ... * kx floats (also enough for the row-major fp32 mel of other paths).
constexpr int kTcMaxClasses = 8;   // FC columns the tensor-core recurrent kernel keeps per thread (gru_tc.cu)
// The tensor-core recurrent kernel serves models of up to kTcMaxClasses classes; wider FC layers run on the exact fp32
// kernel whatever the requested precision (never a silently truncated softmax).
inline bool model_uses_tc(const kws_model* m) {
  return !m->octbit && m->precision == KWS_PRECISION_TC_FP16 && m->cfg.num_classes <= kTcMaxClasses && m->tc_fits;
}
inline bool mel_can_tile(const kws_model* m) { return model_uses_tc(m); }
inline size_t mel_scratch_elems(int64_t S, int32_t n, int n_mel) {
  return static_cast<size_t>(ceil_div(S, 128) * 128) * static_cast<size_t>(n > 0 ? n : 1) * ((n_mel + 15) / 16 * 16);
}
// layer-0 operand geometry of the tiled mel scratch: chunks of 8 mels per half, and whether the lo half exists
inline int mel_tile_chunks(const kws_model* m) { return m->layer[0].tc_kx / 8; }
inline bool mel_tile_split(const kws_model* m) { return m->layer[0].tc_kxw != m->layer[0].tc_kx; }
bool gru_tc_can_split(int in_dim, bool last, int device);                // gru_tc.cu
bool gru_tc_layer_fits(int in_dim, bool split, bool last, int device);
// Stream s gets min(frames_of(head_len + body length), max_frames) frames.  With src.lengths, frames of a stream past
// its own length are zero rows of mel_out.  With src.lengths or pre, nframes_out receives every stream's frame count:
// the seq_len of the recurrent kernels.
int launch_frontend(const kws_model* m, const PcmSource& src, int64_t S, int32_t max_frames, float* mel_out,
                    cudaStream_t st, const FrontendPre* pre = nullptr, bool tiled_out = false,
                    int32_t* nframes_out = nullptr);

struct GruArgs {
  const float* x = nullptr;       // layer-0 input [S, n, M] row-major, or stream-tiled when x_tiled
  bool x_tiled = false;           // mel_tiled_offset layout (tensor-core path, M % 4 == 0)
  int64_t S = 0;
  int32_t n = 0;
  const int32_t* seq_len = nullptr;       // [S] or null
  const uint8_t* zero_state = nullptr;    // [S] or null: 1 = treat incoming state as zero
  const float* state_in = nullptr;        // [layers, S, H]
  float* state_out = nullptr;             // [layers, S, H]
  float* probs = nullptr;                 // [S, n, C]
  float* logits = nullptr;                // [S, n, C] or null
  float* seq_scratch = nullptr;           // inter-layer hand-off of seq_scratch_elems() floats; null -> the model's own
  float* y_rows_scratch = nullptr;        // octbit graph: [S, n, H] last-layer outputs for the FC; null -> the model's own
};
inline size_t seq_scratch_elems(int64_t S, int32_t n, int num_layers) {
  if (num_layers < 2) return 0;
  return static_cast<size_t>(ceil_div(S, 128) * 2) * (n > 0 ? n : 1) * kHidden * 64 * (num_layers > 2 ? 2 : 1);
}
int launch_gru(kws_model* m, const GruArgs& a, cudaStream_t st);        // dispatches on m->precision
int launch_gru_fp32(kws_model* m, const GruArgs& a, cudaStream_t st);   // gru.cu   (exact fp32 FFMA)
int launch_gru_tc(kws_model* m, const GruArgs& a, cudaStream_t st);     // gru_tc.cu (tcgen05, fp16 operands)
int launch_gru_octbit(kws_model* m, const GruArgs& a, cudaStream_t st); // gru_octbit.cu (the octbit-rewritten graph)
int launch_gru_fp32_layer(kws_model* m, const GruArgs& a, int l, const float* x_tiled, float* y_tiled, float* y_rows,
                          cudaStream_t st);                             // gru.cu: one fp32 layer without the FC
void free_octbit(kws_model* m);

}  // namespace kws
