// The stream object behind kws_stream_* (stream.cu), shared with the wave server (server.cu).
#pragma once

#include "common.cuh"
#include "decode_core.cuh"

struct kws_stream {
  kws_model* model = nullptr;
  int device = 0;           // cached: destroy must not dereference the model (it may already be gone)
  kws_stream_config cfg;
  int64_t S = 0;
  int max_frames = 0;       // frames a chunk of cfg.max_chunk samples can produce
  int fpad = 0;             // token slots per window entry (multiple of 16)
  kws::dec::Keyword kw;
  float* state = nullptr;           // [L, S, H]
  int16_t* tail[2] = {nullptr, nullptr};     // [S, 400] ping-pong
  int32_t* tail_len[2] = {nullptr, nullptr}; // [S]
  int cur = 0;
  unsigned char* silence = nullptr; // [S] 1 = VAD said silence for the current chunk
  int32_t* nframes = nullptr;       // [S]
  float* mel = nullptr;             // [S, max_frames, M]
  float* seq = nullptr;             // inter-layer hand-off, private so that stream objects can run concurrently
  float* y_rows = nullptr;          // octbit graph only: [S, max_frames, H] last-layer outputs for the FC
  float* probs = nullptr;           // [S, max_frames, C]
  signed char* tok = nullptr;       // [S, W, fpad]
  unsigned char* slot_frames = nullptr;  // [S, W]
  int32_t* win_head = nullptr;      // [S] oldest slot
  int32_t* win_n = nullptr;         // [S] slots in use
  int32_t* trigger = nullptr;       // [S]
  // host-buffer path: double-buffered staging + private copy stream
  int16_t* pcm_dev[2] = {nullptr, nullptr};
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t copied[2] = {nullptr, nullptr};
  cudaEvent_t consumed[2] = {nullptr, nullptr};
  int host_buf = 0;
  bool consumed_valid[2] = {false, false};
};

namespace kws {

// Per-stream records (kws_stream_export / kws_stream_import, include/kws_b200.h): where the record kernels find the
// carried state of one stream object.  tail / tail_len are the ping-pong half the next step reads (index cur).
struct RecordSlots {
  float* state = nullptr;
  int16_t* tail = nullptr;
  int32_t* tail_len = nullptr;
  signed char* tok = nullptr;
  unsigned char* slot_frames = nullptr;
  int32_t* win_head = nullptr;
  int32_t* win_n = nullptr;
};
RecordSlots record_slots(const kws_stream* st);
int64_t record_bytes(const kws_stream* st);
// Records of ids in [0, total).  table == nullptr: the ids are streams of `st` itself (total = st->S).  Otherwise id g
// is stream g % st->S of the object table[g / st->S] (DEVICE), every object laid out as `st`.
int launch_record_export(const kws_stream* st, const RecordSlots* table, int64_t total, const int64_t* ids, int64_t n,
                         void* records, cudaStream_t cs);
int launch_record_import(const kws_stream* st, const RecordSlots* table, int64_t total, const int64_t* ids, int64_t n,
                         const void* records, int32_t* status_out, cudaStream_t cs);

}  // namespace kws

