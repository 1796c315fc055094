// C-ABI glue: errors, model handle, and the forward entry points (include/kws_b200.h).
#include <cmath>
#include <cstring>
#include <vector>

#include <cuda_fp16.h>

#include "common.cuh"

namespace kws {

static thread_local std::string g_last_error;

void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
}
void clear_error() { g_last_error.clear(); }
int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

int sm_count() {
  static thread_local int cached_dev = -1;
  static thread_local int cached = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev != cached_dev) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached = n;
    cached_dev = dev;
  }
  return cached;
}

template <typename T>
static int upload(T** dst, const T* host, size_t n) {
  *dst = nullptr;
  if (n == 0) return KWS_OK;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(dst), sizeof(T) * n);
  if (e != cudaSuccess) return fail(KWS_ERR_ALLOC, "cudaMalloc(%zu) failed: %s", sizeof(T) * n, cudaGetErrorString(e));
  KWS_CUDA_OK(cudaMemcpy(*dst, host, sizeof(T) * n, cudaMemcpyHostToDevice));
  return KWS_OK;
}

void pack_tc_weights(const float* gates_kernel, const float* cand_kernel, int in_dim, bool split, std::vector<__half>* out,
                     int* kx_out, int* kxw_out);

static void free_model(kws_model* m) {
  if (!m) return;
  cudaFree(m->mel_basis);
  cudaFree(m->mel.quads);
  free_frontend_tc_tables(m);
  cudaFree(m->twiddle400);
  for (int l = 0; l < kMaxLayers; ++l) {
    cudaFree(m->layer[l].gates_kernel);
    cudaFree(m->layer[l].gates_bias);
    cudaFree(m->layer[l].cand_kernel);
    cudaFree(m->layer[l].cand_bias);
    cudaFree(m->layer[l].tc_wpack);
    cudaFree(m->layer[l].tc_bias);
  }
  cudaFree(m->fc_w);
  cudaFree(m->fc_b);
  for (cudaEvent_t e : m->aux_events) cudaEventDestroy(e);
  if (m->aux_stream) cudaStreamDestroy(m->aux_stream);
  cudaFree(m->scratch_mel);
  cudaFree(m->scratch_seq);
  cudaFree(m->scratch_nfr);
  cudaFree(m->tc_xt);
  free_octbit(m);
  delete m;
}

}  // namespace kws

using namespace kws;

extern "C" const char* kws_last_error(void) { return g_last_error.c_str(); }
extern "C" int kws_abi_version(void) { return KWS_B200_ABI_VERSION; }

extern "C" int kws_device_count(void) {
  clear_error();
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) return fail(KWS_ERR_CUDA, "cudaGetDeviceCount failed: %s", cudaGetErrorString(e));
  return n;
}

extern "C" int kws_model_create(const kws_model_config* cfg, const kws_model_weights* w, int device,
                                kws_model** out) {
  clear_error();
  KWS_REQUIRE(cfg && w && out, "NULL argument");
  *out = nullptr;
  KWS_REQUIRE(cfg->hidden == kHidden, "hidden_size must be %d (config/rnn_config.py:84)", kHidden);
  KWS_REQUIRE(cfg->num_layers >= 1 && cfg->num_layers <= kMaxLayers, "num_layers must be in [1, %d]", kMaxLayers);
  KWS_REQUIRE(cfg->num_classes >= 2 && cfg->num_classes <= kMaxClasses, "num_classes must be in [2, %d]", kMaxClasses);
  KWS_REQUIRE(cfg->n_mel >= 1 && cfg->n_mel <= kMaxMel, "n_mel must be in [1, %d]", kMaxMel);
  KWS_REQUIRE(cfg->fft_size == kFft && cfg->hop_size == kHop,
              "the front end is built for fft_size=%d hop_size=%d (config/rnn_config.py:57-58)", kFft, kHop);
  KWS_REQUIRE(w->mel_basis && w->fc_w && w->fc_b, "NULL weight pointer");
  for (int l = 0; l < cfg->num_layers; ++l)
    KWS_REQUIRE(w->gates_kernel[l] && w->gates_bias[l] && w->cand_kernel[l] && w->cand_bias[l],
                "NULL weight pointer for layer %d", l);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0)
    return fail(KWS_ERR_CUDA, "no CUDA device available (%s); libkws_b200 has no CPU fallback",
                e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
  KWS_REQUIRE(device >= 0 && device < ndev, "device %d out of range [0, %d)", device, ndev);
  KWS_CUDA_OK(cudaSetDevice(device));

  kws_model* m = new kws_model();
  m->cfg = *cfg;
  m->device = device;
  m->frontend = default_frontend();
  const int M = cfg->n_mel, H = kHidden, C = cfg->num_classes;
  int rc = upload(&m->mel_basis, w->mel_basis, static_cast<size_t>(kBins) * M);
  {
    // non-zero part of the basis as balanced per-warp quad lists (exact for any basis: zeros contribute nothing)
    std::vector<kws::MelQuad> quads;
    kws::build_mel_quads(w->mel_basis, M, &quads, &m->mel.quads_per_warp);
    if (rc == KWS_OK) rc = upload(&m->mel.quads, quads.data(), quads.size());
  }
  if (rc == KWS_OK) rc = build_frontend_tc_tables(m, w->mel_basis);
  std::vector<float2> tw(20 * 52);          // periodic k2-major table of W400^(n1*k2) (fft400.cuh: kTwStride = 52)
  for (int k2 = 0; k2 < 20; ++k2)
    for (int j = 0; j < 52; ++j) {
      const double a = -2.0 * M_PI * static_cast<double>((j % 20) * k2) / kFft;
      tw[k2 * 52 + j] = make_float2(static_cast<float>(std::cos(a)), static_cast<float>(std::sin(a)));
    }
  if (rc == KWS_OK) rc = upload(&m->twiddle400, tw.data(), tw.size());
  for (int l = 0; l < cfg->num_layers && rc == KWS_OK; ++l) {
    const int in = l == 0 ? M : H;
    m->layer[l].in_dim = in;
    rc = upload(&m->layer[l].gates_kernel, w->gates_kernel[l], static_cast<size_t>(in + H) * 2 * H);
    if (rc == KWS_OK) rc = upload(&m->layer[l].gates_bias, w->gates_bias[l], 2 * H);
    if (rc == KWS_OK) rc = upload(&m->layer[l].cand_kernel, w->cand_kernel[l], static_cast<size_t>(in + H) * H);
    if (rc == KWS_OK) rc = upload(&m->layer[l].cand_bias, w->cand_bias[l], H);
    if (rc == KWS_OK) {
      std::vector<__half> packed;
      // the unbounded mel input is split into hi/lo fp16 operands when the wider weights still fit (gru_tc.cu)
      const bool last = l == cfg->num_layers - 1;
      const bool split = l == 0 && in <= 64 && gru_tc_can_split(in, last, device);
      if (l == 0 && !gru_tc_layer_fits(in, split, last, device)) m->tc_fits = false;   // (very wide inputs) the model then runs the fp32 kernel
      pack_tc_weights(w->gates_kernel[l], w->cand_kernel[l], in, split, &packed, &m->layer[l].tc_kx, &m->layer[l].tc_kxw);
      __half* dptr = nullptr;
      rc = upload(&dptr, packed.data(), packed.size());
      m->layer[l].tc_wpack = dptr;
      std::vector<float> fused(3 * H);
      for (int i = 0; i < 2 * H; ++i) fused[i] = w->gates_bias[l][i];
      for (int i = 0; i < H; ++i) fused[2 * H + i] = w->cand_bias[l][i];
      if (rc == KWS_OK) rc = upload(&m->layer[l].tc_bias, fused.data(), fused.size());
    }
  }
  if (rc == KWS_OK) rc = upload(&m->fc_w, w->fc_w, static_cast<size_t>(H) * C);
  if (rc == KWS_OK) rc = upload(&m->fc_b, w->fc_b, C);
  m->fc_w_host.assign(w->fc_w, w->fc_w + static_cast<size_t>(H) * C);
  m->fc_b_host.assign(w->fc_b, w->fc_b + C);
  if (rc != KWS_OK) {
    free_model(m);
    return rc;
  }
  *out = m;
  return KWS_OK;
}

extern "C" int kws_model_destroy(kws_model* m) {
  clear_error();
  if (m) {
    cudaSetDevice(m->device);
    free_model(m);
  }
  return KWS_OK;
}

extern "C" int kws_model_set_precision(kws_model* m, int precision) {
  clear_error();
  KWS_REQUIRE(m != nullptr, "model is NULL");
  KWS_REQUIRE(precision == KWS_PRECISION_FP32 || precision == KWS_PRECISION_TC_FP16, "unknown precision %d", precision);
  m->precision = precision;
  return KWS_OK;
}

extern "C" int kws_model_get_precision(const kws_model* m) { return m ? m->precision : -1; }

extern "C" int kws_model_set_frontend(kws_model* m, int frontend) {
  clear_error();
  KWS_REQUIRE(m != nullptr, "model is NULL");
  KWS_REQUIRE(frontend == KWS_FRONTEND_FFT || frontend == KWS_FRONTEND_TC, "unknown frontend %d", frontend);
  m->frontend = frontend;
  return KWS_OK;
}

extern "C" int kws_model_get_frontend(const kws_model* m) { return m ? m->frontend : -1; }

namespace kws {
int launch_gru(kws_model* m, const GruArgs& a, cudaStream_t st) {
  if (m->octbit) return launch_gru_octbit(m, a, st);
  return model_uses_tc(m) ? launch_gru_tc(m, a, st) : launch_gru_fp32(m, a, st);
}
}  // namespace kws

extern "C" int kws_num_frames(const kws_model* m, int64_t L) {
  const int fft = m ? m->cfg.fft_size : kFft, hop = m ? m->cfg.hop_size : kHop;
  // 1 + floor((L - fft) / hop) with floor toward -inf (utils/stft.py:60-61)
  const int64_t d = L - fft;
  const int64_t q = d >= 0 ? d / hop : -((-d + hop - 1) / hop);
  return static_cast<int>(1 + q);
}

extern "C" int kws_model_reserve(kws_model* m, int64_t max_streams, int32_t max_frames) {
  KWS_REQUIRE(m != nullptr, "model is NULL");
  if (max_streams <= m->cap_streams && max_frames <= m->cap_frames) return KWS_OK;
  const int64_t S = max_streams > m->cap_streams ? max_streams : m->cap_streams;
  const int32_t n = max_frames > m->cap_frames ? max_frames : m->cap_frames;
  KWS_CUDA_OK(cudaSetDevice(m->device));
  KWS_CUDA_OK(cudaDeviceSynchronize());      // nobody may still be using the old scratch
  cudaFree(m->scratch_mel);
  cudaFree(m->scratch_seq);
  cudaFree(m->scratch_nfr);
  m->scratch_mel = m->scratch_seq = nullptr;
  m->scratch_nfr = nullptr;
  m->cap_streams = 0;
  m->cap_frames = 0;
  const size_t mel_elems = mel_scratch_elems(S, n, m->cfg.n_mel);
  const size_t seq_elems = seq_scratch_elems(S, n, m->cfg.num_layers);
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&m->scratch_mel), sizeof(float) * (mel_elems ? mel_elems : 1));
  if (e == cudaSuccess && m->cfg.num_layers > 1)
    e = cudaMalloc(reinterpret_cast<void**>(&m->scratch_seq), sizeof(float) * (seq_elems ? seq_elems : 1));
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&m->scratch_nfr), sizeof(int32_t) * (S > 0 ? S : 1));
  if (e != cudaSuccess) {
    cudaFree(m->scratch_mel);
    cudaFree(m->scratch_seq);
    m->scratch_mel = m->scratch_seq = nullptr;
    return fail(KWS_ERR_ALLOC, "scratch allocation for %lld streams x %d frames failed: %s",
                static_cast<long long>(S), n, cudaGetErrorString(e));
  }
  m->cap_streams = S;
  m->cap_frames = n;
  return KWS_OK;
}

static int check_pcm(const void* pcm, int dtype, int64_t S, int64_t L, int64_t ld) {
  KWS_REQUIRE(dtype == KWS_PCM_F32 || dtype == KWS_PCM_I16, "unknown pcm dtype %d", dtype);
  KWS_REQUIRE(S >= 0 && L >= 0, "negative size");
  KWS_REQUIRE(ld >= L, "ld_pcm (%lld) < L (%lld)", static_cast<long long>(ld), static_cast<long long>(L));
  KWS_REQUIRE(L < (1LL << 30), "signal too long");
  KWS_REQUIRE(pcm != nullptr || S == 0 || L == 0, "pcm is NULL");
  return KWS_OK;
}

extern "C" int kws_frontend_mel(kws_model* m, const void* pcm, int pcm_dtype, int64_t S, int64_t L,
                                int64_t ld_pcm, float* mel_out, void* stream) {
  return kws_frontend_mel_lens(m, pcm, pcm_dtype, S, L, ld_pcm, nullptr, mel_out, stream);
}

extern "C" int kws_frontend_mel_lens(kws_model* m, const void* pcm, int pcm_dtype, int64_t S, int64_t L, int64_t ld_pcm,
                                     const int32_t* lengths, float* mel_out, void* stream) {
  clear_error();
  KWS_REQUIRE(m != nullptr, "model is NULL");
  int rc = check_pcm(pcm, pcm_dtype, S, L, ld_pcm);
  if (rc != KWS_OK) return rc;
  const int n = kws_num_frames(m, L);
  if (S == 0 || n <= 0) return KWS_OK;
  KWS_REQUIRE(mel_out != nullptr, "mel_out is NULL");
  KWS_CUDA_OK(cudaSetDevice(m->device));
  PcmSource src;
  src.body = pcm;
  src.ld_body = ld_pcm;
  src.body_len = static_cast<int32_t>(L);
  src.body_dtype = pcm_dtype;
  src.lengths = lengths;
  return launch_frontend(m, src, S, n, mel_out, static_cast<cudaStream_t>(stream));
}

extern "C" int kws_gru_forward(kws_model* m, const float* mel, int64_t S, int32_t n, const int32_t* seq_len,
                               const float* state_in, float* probs_out, float* state_out, float* logits_out,
                               void* stream) {
  clear_error();
  KWS_REQUIRE(m != nullptr, "model is NULL");
  KWS_REQUIRE(S >= 0 && n >= 0, "negative size");
  if (S == 0) return KWS_OK;
  KWS_REQUIRE(state_in && state_out, "state pointer is NULL");
  KWS_REQUIRE(n == 0 || (mel && probs_out), "mel / probs_out is NULL");
  KWS_REQUIRE(reinterpret_cast<uintptr_t>(mel) % 16 == 0 && reinterpret_cast<uintptr_t>(state_in) % 16 == 0 &&
                  reinterpret_cast<uintptr_t>(state_out) % 16 == 0,
              "mel / state pointers must be 16-byte aligned");
  KWS_CUDA_OK(cudaSetDevice(m->device));
  GruArgs a;
  a.x = mel;
  a.S = S;
  a.n = n;
  a.seq_len = seq_len;
  a.state_in = state_in;
  a.state_out = state_out;
  a.probs = probs_out;
  a.logits = logits_out;
  return launch_gru(m, a, static_cast<cudaStream_t>(stream));
}

namespace kws {
// Rows t >= seq_len[s] of probs / logits [S, n, C] -> 0 (the recurrent kernels give them the dynamic_rnn value,
// softmax of the bias).  One thread per (stream, frame).
__global__ void zero_past_len_kernel(float* probs, float* logits, long S, int n, int C, const int32_t* seq_len) {
  const long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  if (i >= S * n) return;
  const long s = i / n;
  if (static_cast<int>(i - s * n) < __ldg(seq_len + s)) return;
  for (int c = 0; c < C; ++c) {
    probs[i * C + c] = 0.0f;
    if (logits) logits[i * C + c] = 0.0f;
  }
}
}  // namespace kws

extern "C" int kws_deploy_forward(kws_model* m, const void* pcm, int pcm_dtype, int64_t S, int64_t L,
                                  int64_t ld_pcm, const float* state_in, float* probs_out, float* state_out,
                                  float* logits_out, void* stream) {
  return kws_deploy_forward_lens(m, pcm, pcm_dtype, S, L, ld_pcm, nullptr, state_in, probs_out, state_out, logits_out,
                                 stream);
}

extern "C" int kws_deploy_forward_lens(kws_model* m, const void* pcm, int pcm_dtype, int64_t S, int64_t L, int64_t ld_pcm,
                                       const int32_t* lengths, const float* state_in, float* probs_out, float* state_out,
                                       float* logits_out, void* stream) {
  clear_error();
  KWS_REQUIRE(m != nullptr, "model is NULL");
  int rc = check_pcm(pcm, pcm_dtype, S, L, ld_pcm);
  if (rc != KWS_OK) return rc;
  const int n = kws_num_frames(m, L);
  // the reference graph cannot run on fewer than fft_size samples (n <= 0, utils/stft.py:60-61)
  KWS_REQUIRE(n >= 1, "signal of %lld samples is shorter than one %d-sample frame",
              static_cast<long long>(L), m->cfg.fft_size);
  if (S == 0) return KWS_OK;
  rc = kws_model_reserve(m, S, n);
  if (rc != KWS_OK) return rc;
  PcmSource src;
  src.body = pcm;
  src.ld_body = ld_pcm;
  src.body_len = static_cast<int32_t>(L);
  src.body_dtype = pcm_dtype;
  src.lengths = lengths;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  KWS_CUDA_OK(cudaSetDevice(m->device));
  const bool tiled = mel_can_tile(m);
  // with lengths, the front end writes every stream's frame count n_b: the recurrence's seq_len (never read on the host)
  int32_t* nfr = lengths ? m->scratch_nfr : nullptr;
  rc = launch_frontend(m, src, S, n, m->scratch_mel, st, nullptr, tiled, nfr);
  if (rc != KWS_OK) return rc;
  KWS_REQUIRE(state_in && state_out && probs_out, "state / probs pointer is NULL");
  KWS_REQUIRE(reinterpret_cast<uintptr_t>(state_in) % 16 == 0 && reinterpret_cast<uintptr_t>(state_out) % 16 == 0,
              "state pointers must be 16-byte aligned");
  GruArgs a;
  a.x = m->scratch_mel;
  a.x_tiled = tiled;
  a.S = S;
  a.n = n;
  a.seq_len = nfr;
  a.state_in = state_in;
  a.state_out = state_out;
  a.probs = probs_out;
  a.logits = logits_out;
  rc = launch_gru(m, a, st);
  if (rc != KWS_OK || !lengths) return rc;
  const long rows = static_cast<long>(S) * n;
  zero_past_len_kernel<<<static_cast<unsigned>(ceil_div(rows, 256)), 256, 0, st>>>(probs_out, logits_out, S, n,
                                                                                  m->cfg.num_classes, nfr);
  KWS_LAUNCH_OK("zero_past_len_kernel");
  return KWS_OK;
}
