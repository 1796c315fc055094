/* kws_b200 -- C-ABI of the B200-native keyword-spotting hot path.
 *
 * Plain C, plain pointers and sizes.  Unless a function says "host", every data
 * pointer is a DEVICE pointer owned by the caller and every call is
 * stream-ordered on `stream` (a cudaStream_t passed as void*; NULL = the
 * legacy default stream).  No call on the hot path allocates.  All functions
 * return 0 on success or a negative kws_status; the message for the calling
 * thread's last failure is kws_last_error().  There is no CPU fallback: without
 * a CUDA device every compute entry point fails with KWS_ERR_CUDA.
 *
 * Each entry point names the reference interface it replaces (file:line under
 * colinsongf/keyword_spotting).  INTEGRATION.md shows the ctypes binding a
 * maintainer of the reference would add.
 */
#ifndef KWS_B200_H_
#define KWS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KWS_B200_ABI_VERSION 2

typedef enum kws_status {
  KWS_OK = 0,
  KWS_ERR_INVALID_ARGUMENT = -1, /* TF errors::InvalidArgument in the reference ops */
  KWS_ERR_CUDA = -2,             /* CUDA runtime / launch failure, or no device   */
  KWS_ERR_ALLOC = -3,
  KWS_ERR_UNSUPPORTED = -4
} kws_status;

typedef enum kws_pcm_dtype {
  KWS_PCM_F32 = 0, /* float32 already scaled by 2^-15 (detector.py:40-43 output) */
  KWS_PCM_I16 = 1  /* raw little-endian int16; scaled by 2^-15 on load            */
} kws_pcm_dtype;

typedef enum kws_decode_mode {
  KWS_DECODE_CTC = 0,    /* utils/prediction.py:18-62   ctc_decode        */
  KWS_DECODE_CTC2 = 1,   /* utils/prediction.py:65-86   ctc_decode2       */
  KWS_DECODE_STRICT = 2  /* utils/prediction.py:89-108  ctc_decode_strict */
} kws_decode_mode;

/* Thread-local message of the last failing call ("" if none). */
const char* kws_last_error(void);
int kws_abi_version(void);
/* Number of visible CUDA devices, or a negative kws_status. */
int kws_device_count(void);

/* ------------------------------------------------------------------ model
 * The rnn_ctc deployment model, models/rnn_ctc.py:113-166 (DeployModel), with
 * the constants of config/rnn_config.py:57-65,76-84.                          */
typedef struct kws_model kws_model;

typedef struct kws_model_config {
  int32_t n_mel;       /* config.freq_size: 40 (README) or 60 (shipped)         */
  int32_t hidden;      /* 128 -- the only size the kernels are built for        */
  int32_t num_layers;  /* 2                                                     */
  int32_t num_classes; /* 6                                                     */
  int32_t fft_size;    /* 400; any of 16..512 (frame, rfft length)              */
  int32_t hop_size;    /* 160; any of 1..fft_size                               */
} kws_model_config;

/* HOST pointers to fp32 weights in the TF variable layout (row = input index):
 *   mel_basis    [fft/2+1, n_mel]   librosa.filters.mel(...).T, rnn_ctc.py:139-146
 *   gates_kernel [in_l+H, 2H], gates_bias [2H]   GRUCell "gates"    (cols r | u)
 *   cand_kernel  [in_l+H, H],  cand_bias  [H]    GRUCell "candidate"
 *   fc_w [H, C], fc_b [C]                        weightsClasses / biasesClasses
 * in_0 = n_mel, in_l = H for l > 0.  Copied to the device at creation.        */
typedef struct kws_model_weights {
  const float* mel_basis;
  const float* gates_kernel[4];
  const float* gates_bias[4];
  const float* cand_kernel[4];
  const float* cand_bias[4];
  const float* fc_w;
  const float* fc_b;
} kws_model_weights;

/* Arithmetic of the recurrent kernel (K2+K3).
 *   KWS_PRECISION_TC_FP16 (default): tcgen05 tensor cores, fp16 operands, fp32 accumulation and state --
 *     the "fp32-accumulate mode" of the contract (softmax / state within 1e-3 of the fp32 graph).
 *   KWS_PRECISION_FP32: every product in fp32 on the CUDA cores -- the accuracy baseline (~1e-5).        */
typedef enum kws_precision {
  KWS_PRECISION_FP32 = 0,
  KWS_PRECISION_TC_FP16 = 1
} kws_precision;

/* Formulation of the front end (K1) of a 400/160 model.  Both produce the same mel frames (parity tests run on both).
 *   KWS_FRONTEND_FFT (default): packed-real 20x20 FFT on the CUDA cores / shared memory (csrc/frontend.cu).
 *   KWS_FRONTEND_TC: hop-block partial DFTs on tcgen05 with the twiddles in tensor memory (csrc/frontend_tc.cu);
 *     int16 PCM and n_mel <= 64 only -- other inputs run on the FFT kernel.  Same speed on B200, see DESIGN.md.
 * Models of any other fft_size / hop_size run the general front end (csrc/frontend_dft.cu: the real DFT as one
 * tcgen05 product per 128 frames), whatever kws_model_set_frontend says; its fp32 PCM must lie in (-2, 2). */
typedef enum kws_frontend {
  KWS_FRONTEND_FFT = 0,
  KWS_FRONTEND_TC = 1
} kws_frontend;

/* Rejects (KWS_ERR_INVALID_ARGUMENT) fft_size outside [16, 512] and hop_size outside [1, fft_size]. */
int kws_model_create(const kws_model_config* cfg, const kws_model_weights* host_weights,
                     int device, kws_model** out);
int kws_model_set_frontend(kws_model* m, int frontend);
int kws_model_get_frontend(const kws_model* m);
int kws_model_destroy(kws_model* m);
int kws_model_set_precision(kws_model* m, int precision);
int kws_model_get_precision(const kws_model* m);

/* The octbit-rewritten deployment graph (graph_octbit.pb: main.py:357-371, octbit/octbit_graph.py:461-536).  The
 * rewriter turns every MatMul outside cell_0 into OctbitMatMul (octbit_graph.py:218-225): gates and candidate of the
 * upper GRU layers ([in+H] -> 2H and -> H) and the FC (H -> C); cell_0, the mel projection and every BiasAdd /
 * activation stay float.  HOST pointers per converted MatMul: the qint8 Const [out, in] (already transposed), the
 * op's `scale` attr and its `bias` attr [out] (octbit_graph.py:191-215, 527-536).  NULL = that MatMul stays float.
 * The op quantises its input with the min / max of the WHOLE call (octbit_mat_mul_op.cc:90-124); the reference
 * deploys at batch 1, so the range is per stream -- per time step for the GRU MatMuls, per chunk (all frames of the
 * call) for the FC -- and that is what the batched kernels reproduce: S independent batch-1 graphs.
 * After this call every forward of the model (kws_gru_forward, kws_deploy_forward, kws_stream_step, the wave
 * server) runs the octbit graph; NULL switches back to the float graph.  Stream objects created BEFORE the switch
 * share one model-owned scratch and must then be stepped from a single CUDA stream.                            */
typedef struct kws_octbit_weights {
  const int8_t* gates_wq[4];     /* [2H, in+H] */
  float gates_scale[4];
  const float* gates_obias[4];   /* [2H] */
  const int8_t* cand_wq[4];      /* [H, in+H] */
  float cand_scale[4];
  const float* cand_obias[4];    /* [H] */
  const int8_t* fc_wq;           /* [C, H] */
  float fc_scale;
  const float* fc_obias;         /* [C] */
} kws_octbit_weights;

int kws_model_set_octbit(kws_model* m, const kws_octbit_weights* w);
int kws_model_is_octbit(const kws_model* m);

/* utils/stft.py:60-61: 1 + floor((L - fft)/hop); <= 0 when L < fft. */
int kws_num_frames(const kws_model* m, int64_t signal_length);

/* Grow the model-owned scratch so that forwards of up to `max_streams` x
 * `max_frames` run without allocating.  Called implicitly (and synchronously)
 * by the forwards when the scratch is too small.                             */
int kws_model_reserve(kws_model* m, int64_t max_streams, int32_t max_frames);

/* K1 -- fused framing + 400-point real DFT magnitude + mel projection.
 * Replaces tf_frame (utils/stft.py:27-81), abs(rfft) (models/rnn_ctc.py:137)
 * and the mel matmul (models/rnn_ctc.py:139-149).
 *   pcm [S, ld_pcm] (first L samples of each row used)  ->  mel [S, n, n_mel]  */
int kws_frontend_mel(kws_model* m, const void* pcm, int pcm_dtype, int64_t S, int64_t L,
                     int64_t ld_pcm, float* mel_out, void* stream);

/* kws_frontend_mel over rows of their own lengths (kws_frontend_mel is this call with lengths = NULL).
 * lengths: DEVICE int32 [S], valid samples per row, clamped to [0, L]; NULL = L for every row.  Row b has
 * n_b = max(0, kws_num_frames(m, lengths[b])) frames; the row stride stays n = kws_num_frames(m, L).  No sample at or
 * past lengths[b] is used (they are taken as zeros, as past the end of a row alone), so mel rows 0 .. n_b-1 are bit
 * for bit those of kws_frontend_mel on pcm[b, :lengths[b]] alone; rows n_b .. n-1 are zero.                    */
int kws_frontend_mel_lens(kws_model* m, const void* pcm, int pcm_dtype, int64_t S, int64_t L, int64_t ld_pcm,
                          const int32_t* lengths, float* mel_out, void* stream);

/* K2+K3 -- 2-layer TF-GRUCell recurrence with carried state, FC and softmax.
 * Replaces inference1 / inference2 / tf.nn.softmax (models/rnn_ctc.py:156-165,
 * 202-284).  The (mel frames, rnn_state) -> (softmax, rnn_state) form of the
 * deployment call (models/rnn_ctc.py:150-153).
 *   mel [S, n, n_mel]; state_in/out [layers, S, H]; probs/logits [S, n, C]
 *   seq_len [S] int32 or NULL (dynamic_rnn sequence_length semantics: beyond
 *   the length outputs are zero and the state is carried through)
 *   logits_out may be NULL.  state_in may equal state_out.                    */
int kws_gru_forward(kws_model* m, const float* mel, int64_t S, int32_t n,
                    const int32_t* seq_len, const float* state_in, float* probs_out,
                    float* state_out, float* logits_out, void* stream);

/* The whole deployment call: sess.run(['model/softmax:0','model/rnn_states:0'],
 * {'model/inputX:0': pcm, 'model/rnn_initial_states:0': state})
 * (detector.py:190-193), batched over S streams.                             */
int kws_deploy_forward(kws_model* m, const void* pcm, int pcm_dtype, int64_t S, int64_t L,
                       int64_t ld_pcm, const float* state_in, float* probs_out,
                       float* state_out, float* logits_out, void* stream);

/* kws_deploy_forward over rows of their own lengths (kws_deploy_forward is this call with lengths = NULL).
 * lengths: DEVICE int32 [S], valid samples per row, clamped to [0, L]; NULL = L for every row.  L >= fft_size.
 * Row b has n_b = max(0, kws_num_frames(m, lengths[b])) frames (computed on the device, never read on the host);
 * probs / logits keep the row stride n = kws_num_frames(m, L).  For lengths[b] >= fft_size, rows < n_b of probs and
 * logits and the row's state_out are bit for bit those of kws_deploy_forward on pcm[b, :lengths[b]] alone, for every
 * precision, front end and the octbit graph (whose FC range covers the n_b valid frames).  Rows >= n_b are zero; a
 * row with n_b = 0 has state_out = state_in.  No sample at or past lengths[b] is used (NaN there reaches nothing). */
int kws_deploy_forward_lens(kws_model* m, const void* pcm, int pcm_dtype, int64_t S, int64_t L, int64_t ld_pcm,
                            const int32_t* lengths, const float* state_in, float* probs_out, float* state_out,
                            float* logits_out, void* stream);

/* ----------------------------------------------------------------- decode
 * K4 -- batched CTC peak decoders + keyword test (utils/prediction.py:18-118).
 *   probs [S, T, C] fp32; lens [S] int32 or NULL (= T)
 *   labels_out [S, max_labels] int32 in the reference's own output form
 *     [0, l1, 0, l2, 0, ...] padded with -1 (ctc_predict stops at a negative);
 *     may be NULL.  counts_out [S] int32 = 2k+1 (untruncated); may be NULL.
 *   trigger_out [S] int32 = ctc_predict(seq, keyword); may be NULL.
 *   keyword: decimal label string, e.g. "1233" (1..16 digits 1-9).
 *   thres < 0 selects the mode's reference default (0.5 / 0.4 / 0.5).        */
typedef struct kws_decode_params {
  int32_t mode;        /* kws_decode_mode                         */
  int32_t lockout;     /* 3                                       */
  double thres;        /* <0 -> reference default of the mode     */
  double loose_thres;  /* 0.2 (ctc_decode only)                   */
} kws_decode_params;

int kws_ctc_decode(const float* probs, int64_t S, int32_t T, int32_t C, const int32_t* lens,
                   const kws_decode_params* params, const char* keyword, int32_t* labels_out,
                   int32_t max_labels, int32_t* counts_out, int32_t* trigger_out, void* stream);

/* Levenshtein distance of S (reference, hypothesis) label pairs: the integer that wer() divides by len(r)
 * (utils/wer.py:4-41; used by the validation loop main.py:207-217 through WERCalculator, utils/wer.py:80-106).
 *   ref [S, ld_ref] int32 with ref_len [S] valid entries per row, hyp likewise; dist_out [S] int32.
 *   max_len: upper bound of all lengths, <= 254 (the reference's table is uint8, utils/wer.py:8).        */
int kws_edit_distance(const int32_t* ref, const int32_t* ref_len, int64_t ld_ref, const int32_t* hyp,
                      const int32_t* hyp_len, int64_t ld_hyp, int64_t S, int32_t max_len,
                      int32_t* dist_out, void* stream);

/* ----------------------------------------------------------------- server
 * The HotwordDetector.start loop (detector.py:148-209) for S lock-step streams
 * with all per-stream state resident in HBM: GRU state, carried PCM tail
 * (detector.py:179-183), 15-chunk decision window (utils/queue.py, detector.py:122),
 * VAD reset (detector.py:168-177) and trigger reset (detector.py:201-209).   */
typedef struct kws_stream kws_stream;

typedef struct kws_stream_config {
  int64_t n_streams;
  int32_t max_chunk;      /* largest chunk length in samples (4800 = 300 ms)   */
  int32_t window_chunks;  /* 15                                                */
  int32_t vad_threshold;  /* 30: speech iff sum|x|/32768 > threshold           */
  double decode_thres;    /* 0.4 (ctc_decode2 default)                         */
  char keyword[20];       /* "1233"                                            */
} kws_stream_config;

int kws_stream_create(kws_model* m, const kws_stream_config* cfg, kws_stream** out);
int kws_stream_destroy(kws_stream* st);
/* Forget everything (state, tails, windows) for all streams. */
int kws_stream_reset(kws_stream* st, void* stream);

/* One chunk for every stream.  pcm [S, chunk_len] int16 (row stride ld_pcm).
 *   trigger_out [S] int32 (1 = keyword fired this chunk); may be NULL
 *   probs_out  [S, max_frames, C] fp32 softmax of this chunk's frames, or NULL
 *   nframes_out [S] int32 frames produced this chunk, or NULL
 * max_frames = kws_stream_max_frames().                                      */
int kws_stream_step(kws_stream* st, const int16_t* pcm, int32_t chunk_len, int64_t ld_pcm,
                    int32_t* trigger_out, float* probs_out, int32_t* nframes_out, void* stream);

/* Same, HOST buffers: pcm_host should be pinned for async copies; the call
 * enqueues H2D(pcm) -> step -> D2H(trigger) on `stream` and returns without
 * synchronising (sync the stream before reading trigger_host).               */
int kws_stream_step_host(kws_stream* st, const int16_t* pcm_host, int32_t chunk_len,
                         int32_t* trigger_host, void* stream);

int32_t kws_stream_max_frames(const kws_stream* st);
/* Device pointer to the carried GRU state [layers, S, H] (for inspection). */
const float* kws_stream_state(const kws_stream* st);
/* Stream-ordered copy of the carried GRU state into state_out [layers, S, H]. */
int kws_stream_copy_state(kws_stream* st, float* state_out, void* stream);
/* Window decode of every stream as of the last step (labels as kws_ctc_decode). */
int kws_stream_labels(kws_stream* st, int32_t* labels_out, int32_t max_labels,
                      int32_t* counts_out, void* stream);

/* Per-stream records: everything one stream carries from one chunk to the next, as a fixed-size, self-describing
 * byte block, so that chosen streams can be saved, restored, compared or moved to another object or GPU between
 * chunks.  Little-endian; every section is a multiple of 16 bytes (offsets in bytes, L = num_layers, H = hidden,
 * W = window_chunks, Wp = W rounded up to 16, T = the tail capacity max(400, fft_size rounded up to 8)):
 *     0  uint32 magic 0x5253574B ("KWSR"), uint32 version 1, int32 L, int32 H
 *    16  int32 W, int32 fpad (token slots per window entry, a multiple of 16), int32 record bytes, 0
 *    32  int32 tail_len (carried PCM samples, 0..fft_size - 1), int32 win_n (window entries in use, 0..W), 0, 0
 *    48  GRU state [L][H] fp32, raw bits
 *    48 + 512 L           carried PCM tail [T] int16: the first tail_len samples
 *    48 + 512 L + 2T      slot_frames [Wp] uint8: frames of window entry q, oldest entry first
 *    48 + 512 L + 2T + Wp  tokens [W][fpad] int8: per frame of entry q, the above-threshold winner class - 1, or -1
 * record bytes = 48 + 512 L + 2T + Wp + W fpad (2368 at L = 2, W = 15, max_chunk = 4800, fft_size <= 400: T = 400).
 * A record of another tail capacity differs in the record-bytes field of its header.  Records are canonical: every
 * byte that holds no state is zero (samples past tail_len, tokens past slot_frames[q], entries past win_n, padding),
 * so the record of a stream does not depend on where its window ring starts, and export -> import -> export gives
 * the same bytes.  Per-chunk scratch (VAD flags, frame counts, triggers, mel, probabilities) is not state: each step
 * writes it before reading it.
 *
 * ids: DEVICE int64 [n]; records: DEVICE [n, kws_stream_record_bytes()], 16-byte aligned.  Both calls are
 * stream-ordered, do not allocate and cost O(n), whatever the number of streams.  Ids must be distinct: with a
 * duplicate id, which of its records lands is unspecified.
 * Export of an id outside [0, n_streams) writes an all-zero record, which import rejects.
 * Import treats every record as input from outside the program (it may come from disk).  status_out: DEVICE int32
 * [n] or NULL; 0 = imported, 1 = id outside [0, n_streams), 2 = header does not match this object (magic, version,
 * L, H, W, fpad or record bytes), 3 = malformed field (tail_len outside [0, fft_size - 1], win_n outside [0, W], a used
 * slot_frames above kws_stream_max_frames(), a used token outside [-1, num_classes - 3]).  A rejected record
 * leaves its stream untouched.  An imported stream continues bit for bit as the exported one would have.        */
int64_t kws_stream_record_bytes(const kws_stream* st);
int kws_stream_export(kws_stream* st, const int64_t* ids, int64_t n, void* records, void* stream);
int kws_stream_import(kws_stream* st, const int64_t* ids, int64_t n, const void* records,
                      int32_t* status_out, void* stream);

/* ----------------------------------------------------------------- wave server
 * The serving loop itself (HotwordDetector.start, detector.py:148-212: read a chunk -> model -> decode -> react,
 * forever) for all the streams of one GPU.  The streams are split into `waves` equal groups; a wave is one
 * kws_stream with its own CUDA stream, two pinned HOST ingest slots and, captured at creation, a CUDA graph of the
 * whole chunk:  H2D(pcm) -> front end -> GRU x layers -> decode/trigger -> D2H(trigger flags).  Serving a wave's
 * chunk is one graph launch; waves overlap each other's copies and kernels; a chunk's latency (host clock, submit ->
 * trigger flags visible on the host) is recorded for every (wave, chunk).  One host thread drives a server.       */
typedef struct kws_server kws_server;

typedef struct kws_server_config {
  int64_t n_streams;       /* streams served by this GPU; a multiple of `waves`            */
  int32_t waves;           /* 16: groups served independently                               */
  int32_t chunk_samples;   /* 4800 = 300 ms (README.md:88, detector.py:150)                 */
  int32_t use_graphs;      /* 1: replay CUDA graphs; 0: enqueue copies and kernels directly */
  kws_stream_config stream;/* window / VAD / threshold / keyword (n_streams, max_chunk ignored) */
} kws_server_config;

int kws_server_create(kws_model* m, const kws_server_config* cfg, kws_server** out);
int kws_server_destroy(kws_server* s);
int kws_server_info(const kws_server* s, int64_t* streams_per_wave, int32_t* waves, int32_t* graphs);
/* Forget GRU state, tails and windows of every stream (nothing may be in flight). */
int kws_server_reset(kws_server* s);
/* Pinned HOST buffer [streams_per_wave, chunk_samples] int16 that the NEXT kws_server_submit(wave) will send:
 * the producer (network / audio threads) writes the wave's chunk here.  At most two chunks per wave are in
 * flight, so the slot returned after a submit is free as soon as the chunk before last has been waited for.   */
int16_t* kws_server_ingest_slot(kws_server* s, int32_t wave);
/* Enqueue the wave's chunk (non-blocking). */
int kws_server_submit(kws_server* s, int32_t wave);
/* Block until the wave's oldest chunk in flight is done.  *trigger_host: pinned HOST flags [streams_per_wave]
 * (1 = keyword fired in this chunk; valid until two more submits of the wave); *latency_ms: submit -> now.     */
int kws_server_wait(kws_server* s, int32_t wave, const int32_t** trigger_host, double* latency_ms);
/* `rounds` chunks for every wave from the ingest slots as they are, wave by wave, at most `depth` waves in flight
 * (the steady-state loop of a server whose producers keep the slots filled).                                   */
int kws_server_serve(kws_server* s, int32_t rounds, int32_t depth);
/* Latency percentiles over the chunks completed since the last reset of the statistics, their number, and the
 * number of triggers they raised.  Any output may be NULL.                                                     */
int kws_server_stats(kws_server* s, int reset, double* p50_ms, double* p99_ms, double* max_ms, int64_t* chunks,
                     int64_t* triggers);
/* 1: submit only moves the bytes (H2D of the slot, D2H of the flags) -- the link ceiling of this box for the
 * same buffers, CUDA streams and schedule.  Nothing may be in flight when switching.                           */
int kws_server_set_copy_only(kws_server* s, int copy_only);
/* The wave's stream object (for kws_stream_labels / kws_stream_copy_state); owned by the server. */
kws_stream* kws_server_wave_stream(kws_server* s, int32_t wave);
/* kws_stream_export / kws_stream_import over the server's global stream ids [0, n_streams) (wave = id /
 * streams_per_wave), records of kws_stream_record_bytes(kws_server_wave_stream(s, 0)) bytes.  Nothing may be in
 * flight.  All ids go in one launch; the call synchronises `stream` before returning, so the next
 * kws_server_submit sees the imported state.  The captured graphs stay valid: import writes the buffers they
 * read.                                                                                                        */
int kws_server_export(kws_server* s, const int64_t* ids, int64_t n, void* records, void* stream);
int kws_server_import(kws_server* s, const int64_t* ids, int64_t n, const void* records, int32_t* status_out,
                      void* stream);

/* ----------------------------------------------------------------- octbit
 * K5 -- OctbitMatMul (octbit/octbit_mat_mul_op.cc:49-183; Python wrapper
 * octbit/octbit_ops.py:17-26; op def octbit/octbit_ops_reg.cc:7-15).
 *   x [A, K] fp32, w [B, K] int8 (already transposed), bias [B] fp32
 *   out [A, B] fp32 -- bit-exact with the reference kernel, including the
 *   int16 pair saturation of _mm_maddubs_epi16 and the fp32 epilogue order.
 * Argument checks follow the op: transpose_b must be 1, transpose_a 0, scale > 0
 * (:41-46); K % 64 == 0 (:65-67); w 32-byte aligned (:56-57).
 * workspace: kws_octbit_workspace_bytes(A, K) bytes of device scratch.       */
size_t kws_octbit_workspace_bytes(int64_t A, int64_t K);
int kws_octbit_matmul(const float* x, const int8_t* w, const float* bias, float scale,
                      int transpose_a, int transpose_b, int64_t A, int64_t B, int64_t K,
                      float* out, void* workspace, size_t workspace_bytes, void* stream);

/* Same contract, but always through the exact CUDA-core back end (every pair formed and
 * saturated, four lanes kept apart).  kws_octbit_matmul uses it itself for K > 512; it is
 * exported so tests can hold the tensor-core back end against it.                       */
int kws_octbit_matmul_exact(const float* x, const int8_t* w, const float* bias, float scale,
                            int64_t A, int64_t B, int64_t K, float* out, void* workspace,
                            size_t workspace_bytes, void* stream);

/* octize_weight_int8_signed (octbit/octbit_graph.py:191-215) on the device:
 *   weight [in, out] fp32 -> wq_t [out, in] int8, *scale_host, bias [out] fp32.
 * Synchronises `stream` to return the scale.                                 */
int kws_octize_weight(const float* weight, int64_t in_dim, int64_t out_dim, int8_t* wq_t,
                      float* bias, double* scale_host, void* stream);

/* ----------------------------------------------------------------- posenc
 * K6 -- PositionalEncoding (positional_encoding/positional_encoding_op.cc:32-50;
 * wrapper positional_encoding_op.py:23-24).  out [max_position, encoding_size]
 * fp32; for odd encoding_size the last column is left untouched, as in the
 * reference (:45).                                                           */
int kws_positional_encoding(int32_t max_position, int32_t encoding_size, float* out,
                            void* stream);

/* ----------------------------------------------------------------- attention_ctc
 * The attention_ctc deployment forward pass (models/attention_ctc.py:73-128, :215-274; BASELINE config 5), the
 * consumer of the positional_encoding op: combine_frame folding, input dense + positional encoding, num_layers x
 * {8-head self-attention over all T' positions, add + layer_norm over (T', N), relu FFN, add + layer_norm},
 * output dense (+relu) and softmax.  The graph has no padding mask: kws_attention_forward takes utterances of one
 * length, kws_attention_forward_lens utterances of different lengths, each computed as the graph computes it alone. */
typedef struct kws_attention kws_attention;

typedef struct kws_attention_config {
  int32_t n_mel;         /* 60  (config/attention_config.py:67)  */
  int32_t combine_frame; /* 2   (:79)                             */
  int32_t hidden;        /* 128 (:85) -- the only size the kernels are built for */
  int32_t heads;         /* 8   (:84)                             */
  int32_t num_layers;    /* 3   (:80)                             */
  int32_t ffn;           /* 512 (:82)                             */
  int32_t num_classes;   /* 6                                     */
  int32_t use_relu;      /* 1   (:54) relu on the output layer    */
} kws_attention_config;

/* HOST pointers, fp32, dense-layer kernels as [in, out] (the [1,1,in,out] conv kernels of tf.layers.conv2d):
 *   w_in [combine*n_mel, N], b_in [N]; per layer w_qkv [N, 3N], b_qkv [3N], ln1_g/ln1_b [N] (layer_norm after the
 *   attention sub-layer), w_ff1 [N, F], b_ff1 [F], w_ff2 [F, N], b_ff2 [N], ln2_g/ln2_b [N]; w_out [N, C], b_out [C]. */
typedef struct kws_attention_weights {
  const float* w_in;
  const float* b_in;
  const float* w_qkv[8];
  const float* b_qkv[8];
  const float* ln1_g[8];
  const float* ln1_b[8];
  const float* w_ff1[8];
  const float* b_ff1[8];
  const float* w_ff2[8];
  const float* b_ff2[8];
  const float* ln2_g[8];
  const float* ln2_b[8];
  const float* w_out;
  const float* b_out;
} kws_attention_weights;

int kws_attention_create(const kws_attention_config* cfg, const kws_attention_weights* host_weights, int device,
                         kws_attention** out);
int kws_attention_destroy(kws_attention* m);
/* T' = T / combine_frame + 1 for combine_frame > 1 (models/attention_ctc.py:88-90), T' = T for combine_frame == 1. */
int32_t kws_attention_frames(const kws_attention* m, int32_t T);
/* mel [B, T, n_mel] (DEVICE, e.g. from kws_frontend_mel) -> probs_out [B, T', C]; logits_out may be NULL.
 * Precondition: |mel| and every activation stay below 65520, the largest value the fp16 `hi` part of the tensor-core
 * operand splits holds; larger values give inf / NaN.  Front-end mel output stays far below that.              */
int kws_attention_forward(kws_attention* m, const float* mel, int64_t B, int32_t T, float* probs_out,
                          float* logits_out, void* stream);
/* Variable-length batch: utterance b has lens[b] valid mel frames (DEVICE int32 [B]) in the first rows of mel [B, T, n_mel];
 * the rest of its rows is never read.  Rows 0 .. kws_attention_frames(lens[b]) - 1 of probs_out / logits_out [B, T', C]
 * (T' = kws_attention_frames(T)) are bit-identical to kws_attention_forward on that utterance alone with T = lens[b];
 * the remaining rows are zero.  lens values are clamped to [1, T].  lens == NULL: every utterance has T frames.   */
int kws_attention_forward_lens(kws_attention* m, const float* mel, int64_t B, int32_t T, const int32_t* lens,
                               float* probs_out, float* logits_out, void* stream);

/* ----------------------------------------------------------------- self-test
 * One 128 x N x K tensor-core product through the tcgen05 conventions the recurrent kernel builds on
 * (A in TMEM when ss_mode == 0, in shared memory when 1; B in shared memory; fp32 accumulate in TMEM).
 * A [128, K] fp32 DEVICE, B [N, K] fp32 HOST, D [128, N] fp32 DEVICE.  Both operands are rounded to fp16.
 * Synchronises `stream`.                                                                       */
int kws_debug_tc_gemm(const float* A, const float* B_host, float* D, int N, int K, int ss_mode,
                      void* stream);

/* Debug / test: the kernels of kws_attention_forward one at a time, on caller DEVICE buffers (W_host is HOST).  Each
 * call synchronises `stream` and returns KWS_ERR_UNSUPPORTED for a shape the chosen kernel does not take.
 *   att_linear:  Y [rows, N] = act(A [rows, K] W [K, N] + bias [N]) (+ pe [r % Tp, N] when add_pe), act = relu or none;
 *                path 0 = tcgen05 (N % 128 == 0, K % 4 == 0; W packed for this call), 1 = the fp32 FFMA kernel.
 *   att_core:    qkv [B, Tp, 3 * 16 * heads] (q | k | v, head-major inside each) -> out [B, Tp, 16 * heads],
 *                softmax(q k^T / 4) v per (utterance, head); path 0 = tcgen05 (Tp <= 400), 1 = the FFMA kernel.
 *   att_add_layernorm:  y = layer_norm(a + b) over each utterance's [Tp, N], per-channel gamma / beta (N % 4 == 0);
 *                in_smem = 1 keeps a + b in shared memory (Tp * N <= 51,200), 0 reads a and b three times.
 *   The _lens forms take per-utterance row counts lens (DEVICE int32 [B], in T' units, clamped to [1, Tp]; NULL = Tp)
 *   with rows still at stride Tp, as kws_attention_forward_lens runs them: utterance b uses its first lens[b] rows (and
 *   keys) only, and rows at or past lens[b] of `out` / `y` are not written.                                       */
int kws_debug_att_linear(const float* A, const float* W_host, const float* bias, const float* pe, int32_t Tp,
                         int64_t rows, int32_t K, int32_t N, int relu, int add_pe, int path, float* Y, void* stream);
int kws_debug_att_core(const float* qkv, int64_t B, int32_t Tp, int32_t heads, int path, float* out, void* stream);
int kws_debug_att_add_layernorm(const float* a, const float* b, const float* gamma, const float* beta, int64_t B,
                                int32_t Tp, int32_t N, int in_smem, float* y, void* stream);
int kws_debug_att_core_lens(const float* qkv, int64_t B, int32_t Tp, const int32_t* lens, int32_t heads, int path,
                            float* out, void* stream);
int kws_debug_att_add_layernorm_lens(const float* a, const float* b, const float* gamma, const float* beta, int64_t B,
                                     int32_t Tp, const int32_t* lens, int32_t N, int in_smem, float* y, void* stream);

/* Debug: enable/disable and read the phase timeline (SM clock ticks) of the first tile of CTA 0 of the last
 * tensor-core GRU launch; see csrc/gru_tc.cu.  host_out may be NULL (only set the switch).               */
int kws_debug_tc_timeline(int enable, long long* host_out, int count);

/* Debug / test (host only, needs no device): the front end's per-warp mel "quad" lists for a basis [201, n_mel]
 * (csrc/frontend.cu, build_mel_quads).  quads_out receives records of 8 ints {4 weights (float bits), magnitude row byte
 * offset, output band byte offset or -1, 0, 0}, 10 warps x the returned quads-per-warp; quads_out may be NULL.     */
int kws_debug_mel_quads(const float* basis, int n_mel, int* quads_out, int capacity);

/* Debug: per-part device time of kws_stream_step (front end incl. the fused VAD/tail pre-step | GRU layers | decode
 * + trigger), CUDA events on the step's stream.  While enabled every step synchronises; ms_out3 receives the sums
 * over *steps_out steps since it was enabled (either may be NULL).  Switching resets the sums.             */
int kws_debug_step_timing(int enable, double* ms_out3, long long* steps_out);

#ifdef __cplusplus
}
#endif
#endif /* KWS_B200_H_ */
