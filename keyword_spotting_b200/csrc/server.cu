// Wave server: the serving loop of the reference (HotwordDetector.start, detector.py:148-212) at scale.
//
// The reference serves ONE microphone: read a 300 ms chunk, run the model, decode, react to the trigger, repeat.
// Here one GPU serves S streams.  They are split into W waves of S/W streams; a wave is one stream object
// (kws_stream: GRU state, carried tails, decision windows -- all resident in HBM) with its own CUDA stream, two
// pinned host ingest slots (the producer writes chunk k+1 while chunk k is in flight), a device staging buffer per
// slot, and -- captured once at creation -- one CUDA graph per slot parity holding the whole chunk:
//     H2D(pinned PCM) -> front end (+VAD, tail carry) -> GRU layer 0 -> GRU layer 1 (+FC, softmax)
//                     -> window decode + trigger + resets -> D2H(trigger flags)
// so serving a wave's chunk is ONE graph launch.  Waves are independent, so the copies of one wave overlap the
// kernels of another, and a chunk's latency is that of its wave, not of the whole batch.  Latency is accounted per
// (wave, chunk) on the host clock from submit to the moment its trigger flags are visible on the host.
//
// A copy-only mode replays the same graphs without the kernels: the link ceiling of this box for the same buffers,
// streams and schedule, against which the full path is reported (bench.py: e2e / copy_ceiling).
#include <algorithm>
#include <chrono>
#include <cstring>
#include <vector>

#include "stream_internal.cuh"

namespace kws {

using clk = std::chrono::steady_clock;

struct Wave {
  kws_stream* st = nullptr;
  cudaStream_t cs = nullptr;
  int16_t* host_pcm[2] = {nullptr, nullptr};    // pinned ingest slots [Sw, chunk]
  int32_t* host_trig[2] = {nullptr, nullptr};   // pinned trigger flags [Sw]
  int16_t* dev_pcm[2] = {nullptr, nullptr};
  cudaGraphExec_t full[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};   // [slot][tail ping-pong of the stream object]
  cudaGraphExec_t copy[2] = {nullptr, nullptr};
  cudaEvent_t done[2] = {nullptr, nullptr};
  long long submitted = 0, completed = 0;
  clk::time_point t_submit[2];
};

}  // namespace kws

struct kws_server {
  kws_model* model = nullptr;
  int device = 0;
  kws_server_config cfg;
  int64_t Sw = 0;
  int graphs = 0;                   // 1: chunks are served by graph replay
  int copy_only = 0;
  std::vector<kws::Wave> waves;
  std::vector<float> latency_ms;    // one entry per completed (wave, chunk)
  long long triggers = 0;
  kws::RecordSlots* record_table = nullptr;        // DEVICE [waves]: the record kernels' per-wave pointers
  std::vector<kws::RecordSlots> record_table_host;
};

namespace kws {

static void free_server(kws_server* s) {
  if (!s) return;
  cudaSetDevice(s->device);
  cudaDeviceSynchronize();
  for (Wave& w : s->waves) {
    for (int i = 0; i < 2; ++i) {
      for (int c = 0; c < 2; ++c)
        if (w.full[i][c]) cudaGraphExecDestroy(w.full[i][c]);
      if (w.copy[i]) cudaGraphExecDestroy(w.copy[i]);
      if (w.done[i]) cudaEventDestroy(w.done[i]);
      if (w.host_pcm[i]) cudaFreeHost(w.host_pcm[i]);
      if (w.host_trig[i]) cudaFreeHost(w.host_trig[i]);
      cudaFree(w.dev_pcm[i]);
    }
    if (w.st) kws_stream_destroy(w.st);
    if (w.cs) cudaStreamDestroy(w.cs);
  }
  cudaFree(s->record_table);
  delete s;
}

// What one chunk of a wave enqueues on its stream (directly, or once under capture).
static int enqueue_chunk(kws_server* s, Wave& w, int slot, bool with_kernels) {
  const size_t pcm_bytes = sizeof(int16_t) * s->Sw * s->cfg.chunk_samples;
  KWS_CUDA_OK(cudaMemcpyAsync(w.dev_pcm[slot], w.host_pcm[slot], pcm_bytes, cudaMemcpyHostToDevice, w.cs));
  if (with_kernels) {
    const int rc = kws_stream_step(w.st, w.dev_pcm[slot], s->cfg.chunk_samples, s->cfg.chunk_samples, nullptr, nullptr,
                                   nullptr, w.cs);
    if (rc != KWS_OK) return rc;
  }
  KWS_CUDA_OK(cudaMemcpyAsync(w.host_trig[slot], w.st->trigger, sizeof(int32_t) * s->Sw, cudaMemcpyDeviceToHost, w.cs));
  return KWS_OK;
}

static int capture(kws_server* s, Wave& w, int slot, bool with_kernels, cudaGraphExec_t* out) {
  cudaGraph_t graph = nullptr;
  KWS_CUDA_OK(cudaStreamBeginCapture(w.cs, cudaStreamCaptureModeRelaxed));
  const int rc = enqueue_chunk(s, w, slot, with_kernels);
  const cudaError_t e = cudaStreamEndCapture(w.cs, &graph);
  if (rc != KWS_OK) {
    if (graph) cudaGraphDestroy(graph);
    return rc;
  }
  if (e != cudaSuccess) return fail(KWS_ERR_CUDA, "cudaStreamEndCapture failed: %s", cudaGetErrorString(e));
  const cudaError_t e2 = cudaGraphInstantiate(out, graph, 0);
  cudaGraphDestroy(graph);
  if (e2 != cudaSuccess) return fail(KWS_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(e2));
  return KWS_OK;
}

}  // namespace kws

using namespace kws;

extern "C" int kws_server_create(kws_model* m, const kws_server_config* cfg, kws_server** out) {
  clear_error();
  KWS_REQUIRE(m && cfg && out, "NULL argument");
  *out = nullptr;
  KWS_REQUIRE(cfg->waves >= 1 && cfg->waves <= 4096, "waves must be in [1, 4096]");
  KWS_REQUIRE(cfg->n_streams >= cfg->waves && cfg->n_streams % cfg->waves == 0,
              "n_streams (%lld) must be a positive multiple of waves (%d)", static_cast<long long>(cfg->n_streams), cfg->waves);
  KWS_REQUIRE(cfg->chunk_samples >= 1 && cfg->chunk_samples <= (1 << 20), "chunk_samples out of range");
  KWS_CUDA_OK(cudaSetDevice(m->device));
  kws_server* s = new kws_server();
  s->model = m;
  s->device = m->device;
  s->cfg = *cfg;
  s->Sw = cfg->n_streams / cfg->waves;
  s->waves.resize(cfg->waves);
  kws_stream_config sc = cfg->stream;
  sc.n_streams = s->Sw;
  sc.max_chunk = cfg->chunk_samples;
  const size_t pcm_bytes = sizeof(int16_t) * s->Sw * cfg->chunk_samples;
  auto bail = [&](int rc) {
    std::string msg = kws_last_error();
    free_server(s);
    set_error("%s", msg.c_str());
    return rc;
  };
  for (Wave& w : s->waves) {
    int rc = kws_stream_create(m, &sc, &w.st);
    if (rc != KWS_OK) return bail(rc);
    if (cudaStreamCreateWithFlags(&w.cs, cudaStreamNonBlocking) != cudaSuccess)
      return bail(fail(KWS_ERR_CUDA, "cudaStreamCreate failed"));
    for (int i = 0; i < 2; ++i) {
      // (write-combined slots were measured at 8 GPUs: the same 23.3 GB/s per GPU -- the ceiling is the host's, not the cache snoop's)
      cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(&w.host_pcm[i]), pcm_bytes, cudaHostAllocDefault);
      if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void**>(&w.host_trig[i]), sizeof(int32_t) * s->Sw, cudaHostAllocDefault);
      if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&w.dev_pcm[i]), pcm_bytes);
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(&w.done[i], cudaEventDisableTiming);
      if (e != cudaSuccess) return bail(fail(KWS_ERR_ALLOC, "wave buffers (%zu B pinned + device): %s", pcm_bytes, cudaGetErrorString(e)));
      std::memset(w.host_pcm[i], 0, pcm_bytes);
      std::memset(w.host_trig[i], 0, sizeof(int32_t) * s->Sw);
    }
  }
  s->record_table_host.resize(s->waves.size());
  if (cudaMalloc(reinterpret_cast<void**>(&s->record_table), sizeof(RecordSlots) * s->waves.size()) != cudaSuccess)
    return bail(fail(KWS_ERR_ALLOC, "record table of %zu waves", s->waves.size()));
  if (cfg->use_graphs) {
    // Two warm-up chunks per wave outside capture (first-use initialisation of every kernel must not happen under
    // capture), then forget them; then capture every (ingest slot, tail ping-pong) combination: kws_stream_step
    // flips the stream object's ping-pong on the host while it enqueues, so each slot is captured twice in a row.
    for (Wave& w : s->waves) {
      int rc = enqueue_chunk(s, w, 0, true);
      if (rc == KWS_OK) rc = enqueue_chunk(s, w, 1, true);
      if (rc == KWS_OK) rc = kws_stream_reset(w.st, w.cs);
      if (rc != KWS_OK) return bail(rc);
    }
    KWS_CUDA_OK(cudaDeviceSynchronize());
    for (Wave& w : s->waves)
      for (int slot = 0; slot < 2; ++slot) {
        int rc = KWS_OK;
        for (int c = 0; c < 2 && rc == KWS_OK; ++c) rc = capture(s, w, slot, true, &w.full[slot][w.st->cur]);
        if (rc == KWS_OK) rc = capture(s, w, slot, false, &w.copy[slot]);
        if (rc != KWS_OK) return bail(rc);
      }
    s->graphs = 1;
  }
  *out = s;
  return KWS_OK;
}

extern "C" int kws_server_destroy(kws_server* s) {
  clear_error();
  free_server(s);
  return KWS_OK;
}

extern "C" int kws_server_info(const kws_server* s, int64_t* streams_per_wave, int32_t* waves, int32_t* graphs) {
  clear_error();
  KWS_REQUIRE(s != nullptr, "server is NULL");
  if (streams_per_wave) *streams_per_wave = s->Sw;
  if (waves) *waves = static_cast<int32_t>(s->waves.size());
  if (graphs) *graphs = s->graphs;
  return KWS_OK;
}

extern "C" int kws_server_set_copy_only(kws_server* s, int copy_only) {
  clear_error();
  KWS_REQUIRE(s != nullptr, "server is NULL");
  for (const Wave& w : s->waves) KWS_REQUIRE(w.submitted == w.completed, "chunks are in flight");
  s->copy_only = copy_only ? 1 : 0;
  return KWS_OK;
}

extern "C" int16_t* kws_server_ingest_slot(kws_server* s, int32_t wave) {
  if (!s || wave < 0 || wave >= static_cast<int>(s->waves.size())) return nullptr;
  Wave& w = s->waves[wave];
  return w.host_pcm[w.submitted & 1];
}

extern "C" int kws_server_submit(kws_server* s, int32_t wave) {
  clear_error();
  KWS_REQUIRE(s != nullptr, "server is NULL");
  KWS_REQUIRE(wave >= 0 && wave < static_cast<int>(s->waves.size()), "wave %d out of range", wave);
  Wave& w = s->waves[wave];
  KWS_REQUIRE(w.submitted - w.completed < 2, "wave %d already has two chunks in flight: wait first", wave);
  const int slot = static_cast<int>(w.submitted & 1);
  KWS_CUDA_OK(cudaSetDevice(s->device));
  w.t_submit[slot] = clk::now();
  if (s->graphs) {
    KWS_CUDA_OK(cudaGraphLaunch(s->copy_only ? w.copy[slot] : w.full[slot][w.st->cur], w.cs));
    if (!s->copy_only) w.st->cur ^= 1;            // the captured step reads tail[cur] and writes tail[cur ^ 1]
  } else {
    const int rc = enqueue_chunk(s, w, slot, !s->copy_only);
    if (rc != KWS_OK) return rc;
  }
  KWS_CUDA_OK(cudaEventRecord(w.done[slot], w.cs));
  ++w.submitted;
  return KWS_OK;
}

extern "C" int kws_server_wait(kws_server* s, int32_t wave, const int32_t** trigger_host, double* latency_ms) {
  clear_error();
  KWS_REQUIRE(s != nullptr, "server is NULL");
  KWS_REQUIRE(wave >= 0 && wave < static_cast<int>(s->waves.size()), "wave %d out of range", wave);
  Wave& w = s->waves[wave];
  KWS_REQUIRE(w.completed < w.submitted, "wave %d has nothing in flight", wave);
  const int slot = static_cast<int>(w.completed & 1);
  KWS_CUDA_OK(cudaEventSynchronize(w.done[slot]));
  const double ms = std::chrono::duration<double, std::milli>(clk::now() - w.t_submit[slot]).count();
  s->latency_ms.push_back(static_cast<float>(ms));
  ++w.completed;
  if (!s->copy_only) {
    long long n = 0;
    const int32_t* t = w.host_trig[slot];
    for (int64_t i = 0; i < s->Sw; ++i) n += t[i];
    s->triggers += n;
  }
  if (trigger_host) *trigger_host = w.host_trig[slot];
  if (latency_ms) *latency_ms = ms;
  return KWS_OK;
}

extern "C" int kws_server_serve(kws_server* s, int32_t rounds, int32_t depth) {
  clear_error();
  KWS_REQUIRE(s != nullptr, "server is NULL");
  KWS_REQUIRE(rounds >= 0 && depth >= 1, "rounds must be >= 0 and depth >= 1");
  const int W = static_cast<int>(s->waves.size());
  std::vector<int> inflight;                    // FIFO of waves with a chunk in flight
  inflight.reserve(static_cast<size_t>(depth) + 1);
  size_t head = 0;
  auto retire = [&]() -> int {
    const int rc = kws_server_wait(s, inflight[head], nullptr, nullptr);
    ++head;
    if (head > 1024) {
      inflight.erase(inflight.begin(), inflight.begin() + static_cast<long>(head));
      head = 0;
    }
    return rc;
  };
  for (int k = 0; k < rounds; ++k)
    for (int w = 0; w < W; ++w) {
      while (static_cast<int>(inflight.size() - head) >= depth || s->waves[w].submitted - s->waves[w].completed >= 2) {
        const int rc = retire();
        if (rc != KWS_OK) return rc;
      }
      const int rc = kws_server_submit(s, w);
      if (rc != KWS_OK) return rc;
      inflight.push_back(w);
    }
  while (head < inflight.size()) {
    const int rc = retire();
    if (rc != KWS_OK) return rc;
  }
  return KWS_OK;
}

extern "C" int kws_server_stats(kws_server* s, int reset, double* p50_ms, double* p99_ms, double* max_ms,
                                int64_t* chunks, int64_t* triggers) {
  clear_error();
  KWS_REQUIRE(s != nullptr, "server is NULL");
  std::vector<float> v = s->latency_ms;
  std::sort(v.begin(), v.end());
  const size_t n = v.size();
  if (p50_ms) *p50_ms = n ? v[n / 2] : 0.0;
  if (p99_ms) *p99_ms = n ? v[std::min(n - 1, static_cast<size_t>(0.99 * n))] : 0.0;
  if (max_ms) *max_ms = n ? v[n - 1] : 0.0;
  if (chunks) *chunks = static_cast<int64_t>(n);
  if (triggers) *triggers = s->triggers;
  if (reset) {
    s->latency_ms.clear();
    s->triggers = 0;
  }
  return KWS_OK;
}

extern "C" int kws_server_reset(kws_server* s) {
  clear_error();
  KWS_REQUIRE(s != nullptr, "server is NULL");
  KWS_CUDA_OK(cudaSetDevice(s->device));
  for (Wave& w : s->waves) {
    KWS_REQUIRE(w.submitted == w.completed, "chunks are in flight");
    const int rc = kws_stream_reset(w.st, w.cs);
    if (rc != KWS_OK) return rc;
    KWS_CUDA_OK(cudaStreamSynchronize(w.cs));
  }
  return KWS_OK;
}

// The per-wave pointers of the record kernels, as of now: each wave's tail ping-pong half is the one its next chunk
// reads (the captured graphs point at both halves, so writing there keeps them valid).
static int upload_record_table(kws_server* s, cudaStream_t cs) {
  KWS_REQUIRE(s != nullptr, "server is NULL");
  for (const Wave& w : s->waves) KWS_REQUIRE(w.submitted == w.completed, "chunks are in flight");
  KWS_CUDA_OK(cudaSetDevice(s->device));
  for (size_t i = 0; i < s->waves.size(); ++i) s->record_table_host[i] = record_slots(s->waves[i].st);
  KWS_CUDA_OK(cudaMemcpyAsync(s->record_table, s->record_table_host.data(), sizeof(RecordSlots) * s->waves.size(),
                              cudaMemcpyHostToDevice, cs));
  return KWS_OK;
}

extern "C" int kws_server_export(kws_server* s, const int64_t* ids, int64_t n, void* records, void* stream) {
  clear_error();
  cudaStream_t cs = static_cast<cudaStream_t>(stream);
  int rc = upload_record_table(s, cs);
  if (rc == KWS_OK)
    rc = launch_record_export(s->waves[0].st, s->record_table, s->cfg.n_streams, ids, n, records, cs);
  if (rc == KWS_OK) KWS_CUDA_OK(cudaStreamSynchronize(cs));
  return rc;
}

extern "C" int kws_server_import(kws_server* s, const int64_t* ids, int64_t n, const void* records,
                                 int32_t* status_out, void* stream) {
  clear_error();
  cudaStream_t cs = static_cast<cudaStream_t>(stream);
  int rc = upload_record_table(s, cs);
  if (rc == KWS_OK)
    rc = launch_record_import(s->waves[0].st, s->record_table, s->cfg.n_streams, ids, n, records, status_out, cs);
  if (rc == KWS_OK) KWS_CUDA_OK(cudaStreamSynchronize(cs));
  return rc;
}

extern "C" kws_stream* kws_server_wave_stream(kws_server* s, int32_t wave) {
  if (!s || wave < 0 || wave >= static_cast<int>(s->waves.size())) return nullptr;
  return s->waves[wave].st;
}
