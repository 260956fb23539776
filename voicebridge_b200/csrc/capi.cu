// capi.cu — the C ABI of libvbgpu.so (include/vbgpu.h): handle lifetime, host<->device staging, batch layouts and the
// fused PCM -> log-likelihood / statistics pipelines.  Kernels live in frontend.cu, featpipe.cu, score_*.cu, accum.cu.
#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <mutex>

#include "common.h"

namespace vb {

std::string &last_error() {
  static thread_local std::string e;
  return e;
}

int fail(int code, const char *fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  last_error() = buf;
  return code;
}

int num_sms(int device) {
  static std::mutex mu;
  static int cache[64] = {0};
  std::lock_guard<std::mutex> lk(mu);
  if (device < 0 || device >= 64) return 148;
  if (cache[device] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || v <= 0) v = 148;
    cache[device] = v;
  }
  return cache[device];
}

__global__ void fill_frame2utt_kernel(const int64_t *__restrict__ frame_offsets, int32_t n_utts, int64_t total,
                                      int32_t *__restrict__ frame2utt) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    int lo = 0, hi = n_utts;  // last u with frame_offsets[u] <= t
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (frame_offsets[mid] <= t) lo = mid;
      else hi = mid;
    }
    frame2utt[t] = lo;
  }
}

void launch_fill_frame2utt(const int64_t *d_frame_offsets, int32_t n_utts, int64_t total_frames, int32_t *d_frame2utt,
                           cudaStream_t s) {
  if (total_frames == 0) return;
  int64_t blocks = (total_frames + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  fill_frame2utt_kernel<<<(int)blocks, 256, 0, s>>>(d_frame_offsets, n_utts, total_frames, d_frame2utt);
}

int BatchLayout::update(const int64_t *sample_offsets, const int64_t *frame_offsets, int32_t n, const int32_t *utt2spk,
                        const int32_t *utt_aux, cudaStream_t s) {
  auto same64 = [](const std::vector<int64_t> &v, const int64_t *p, size_t k) {
    return p ? (v.size() == k && std::memcmp(v.data(), p, k * 8) == 0) : v.empty();
  };
  auto same32 = [](const std::vector<int32_t> &v, const int32_t *p, size_t k) {
    return p ? (v.size() == k && std::memcmp(v.data(), p, k * 4) == 0) : v.empty();
  };
  if (n == n_utts && n_utts > 0 && same64(h_sample_offsets, sample_offsets, n + 1) &&
      same64(h_frame_offsets, frame_offsets, n + 1) && same32(h_utt2spk, utt2spk, n) && same32(h_utt_aux, utt_aux, n))
    return 0;
  n_utts = n;
  if (sample_offsets) h_sample_offsets.assign(sample_offsets, sample_offsets + n + 1);
  else h_sample_offsets.clear();
  h_frame_offsets.assign(frame_offsets, frame_offsets + n + 1);
  if (utt2spk) h_utt2spk.assign(utt2spk, utt2spk + n);
  else h_utt2spk.clear();
  if (utt_aux) h_utt_aux.assign(utt_aux, utt_aux + n);
  else h_utt_aux.clear();
  total_frames = frame_offsets[n];
  total_samples = sample_offsets ? sample_offsets[n] : 0;
  VB_CUDA(cudaStreamSynchronize(s));  // the staging buffer may still be in flight from the previous layout
  const size_t b64 = (size_t)(n + 1) * 8, b32 = (size_t)(n > 0 ? n : 1) * 4;
  VB_TRY(stage.reserve(2 * b64 + 2 * b32));
  VB_TRY(d_sample_offsets.reserve(b64));
  VB_TRY(d_frame_offsets.reserve(b64));
  VB_TRY(d_utt2spk.reserve(b32));
  VB_TRY(d_utt_aux.reserve(b32));
  VB_TRY(d_frame2utt.reserve((size_t)(total_frames > 0 ? total_frames : 1) * 4));
  char *st = stage.as<char>();
  if (sample_offsets) {
    std::memcpy(st, sample_offsets, b64);
    VB_CUDA(cudaMemcpyAsync(d_sample_offsets.p, st, b64, cudaMemcpyHostToDevice, s));
  }
  std::memcpy(st + b64, frame_offsets, b64);
  VB_CUDA(cudaMemcpyAsync(d_frame_offsets.p, st + b64, b64, cudaMemcpyHostToDevice, s));
  if (utt2spk) {
    std::memcpy(st + 2 * b64, utt2spk, (size_t)n * 4);
    VB_CUDA(cudaMemcpyAsync(d_utt2spk.p, st + 2 * b64, (size_t)n * 4, cudaMemcpyHostToDevice, s));
  }
  if (utt_aux) {
    std::memcpy(st + 2 * b64 + b32, utt_aux, (size_t)n * 4);
    VB_CUDA(cudaMemcpyAsync(d_utt_aux.p, st + 2 * b64 + b32, (size_t)n * 4, cudaMemcpyHostToDevice, s));
  }
  launch_fill_frame2utt(d_frame_offsets.as<int64_t>(), n, total_frames, d_frame2utt.as<int32_t>(), s);
  VB_CUDA(cudaGetLastError());
  return 0;
}

int check_device(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0)
    return fail(VBGPU_ERR_CUDA, "no CUDA device available (%s); libvbgpu has no CPU fallback",
                e == cudaSuccess ? "count=0" : cudaGetErrorString(e));
  if (device < 0 || device >= n) return fail(VBGPU_ERR_INVALID, "device %d out of range [0,%d)", device, n);
  return 0;
}

static int32_t num_frames_of(const vbgpu_mfcc_s *h, int64_t n) {  // feature-window.cc:41-87 (flush semantics)
  if (h->opts.snip_edges) return n < h->L ? 0 : (int32_t)(1 + (n - h->L) / h->shift);
  return (int32_t)((n + h->shift / 2) / h->shift);
}

static bool is_pinned_or_device(const void *p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Host -> device copy of a possibly pageable buffer, then wait (simple synchronous paths).
static int h2d(void *d, const void *h, size_t bytes, cudaStream_t s) {
  if (bytes == 0) return 0;
  VB_CUDA(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, s));
  return 0;
}
static int d2h(void *h, const void *d, size_t bytes, cudaStream_t s) {
  if (bytes == 0) return 0;
  VB_CUDA(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, s));
  return 0;
}

// Resolve per-utterance VTLN factors to mel-table indices, (re)building device tables when a new factor appears.
static int resolve_vtln(vbgpu_mfcc_t h, const float *vtln_warp, int32_t n_utts, std::vector<int32_t> *idx) {
  idx->clear();
  if (!vtln_warp) return 0;
  bool grew = false, any = false;
  idx->resize(n_utts);
  for (int32_t u = 0; u < n_utts; u++) {
    const float w = vtln_warp[u];
    size_t k = 0;
    for (; k < h->warps.size(); k++)
      if (h->warps[k] == w) break;
    if (k == h->warps.size()) {
      if (h->warps.size() >= 64) return fail(VBGPU_ERR_INVALID, "more than 64 distinct VTLN warp factors");
      h->warps.push_back(w);
      grew = true;
    }
    (*idx)[u] = (int32_t)k;
    any |= (k != 0);
  }
  if (grew) VB_TRY(mfcc_build_tables(h));
  if (!any && h->warps.size() == 1) idx->clear();
  return 0;
}

static int mfcc_prepare(vbgpu_mfcc_t h, const int64_t *sample_offsets, int32_t n_utts, const float *vtln_warp,
                        cudaStream_t s) {
  VB_CHECK(n_utts >= 0 && sample_offsets, "null sample_offsets");
  std::vector<int64_t> fo(n_utts + 1, 0);
  for (int32_t u = 0; u < n_utts; u++) {
    const int64_t n = sample_offsets[u + 1] - sample_offsets[u];
    VB_CHECK(n >= 0, "sample_offsets not monotone at utterance %d", u);
    fo[u + 1] = fo[u] + num_frames_of(h, n);
  }
  std::vector<int32_t> mel_idx;
  VB_TRY(resolve_vtln(h, vtln_warp, n_utts, &mel_idx));
  if (h->warps.size() > 1 && mel_idx.empty()) mel_idx.assign(n_utts, 0);
  return h->layout.update(sample_offsets, fo.data(), n_utts, nullptr, mel_idx.empty() ? nullptr : mel_idx.data(), s);
}

}  // namespace vb

using namespace vb;

extern "C" {

int vbgpu_version(void) { return 100; }
const char *vbgpu_last_error(void) { return last_error().c_str(); }

int vbgpu_device_count(int *count) {
  VB_CHECK(count, "null count");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    *count = 0;
    return fail(VBGPU_ERR_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
  }
  *count = n;
  return 0;
}

int vbgpu_debug_live_bytes(int64_t *device_bytes, int64_t *pinned_bytes) {
  VB_CHECK(device_bytes && pinned_bytes, "null argument");
  *device_bytes = live_device_bytes.load();
  *pinned_bytes = live_pinned_bytes.load();
  return 0;
}

// ================================================================================================================
// MFCC
// ================================================================================================================
void vbgpu_mfcc_opts_default(vbgpu_mfcc_opts *o) {
  if (!o) return;
  *o = vbgpu_mfcc_opts{16000.0f, 10.0f, 25.0f, 1.0f, 0.97f, 1, 0, 1, 0.42f, 1, 23, 20.0f, 0.0f, 100.0f, -500.0f, 0, 13,
                       1, 0.0f, 1, 22.0f, 0};
}

int vbgpu_mfcc_create(const vbgpu_mfcc_opts *opts, int device, vbgpu_mfcc_t *out) {
  VB_CHECK(opts && out, "null argument");
  *out = nullptr;
  VB_CHECK(opts->round_to_power_of_two, "round_to_power_of_two=false is not supported");
  VB_CHECK(opts->num_bins >= 3 && opts->num_bins <= 32, "num_bins %d not in [3,32]", opts->num_bins);
  VB_CHECK(opts->num_ceps >= 1 && opts->num_ceps <= opts->num_bins, "num_ceps %d > num_bins %d", opts->num_ceps,
           opts->num_bins);
  VB_CHECK(opts->preemph_coeff >= 0.0f && opts->preemph_coeff <= 1.0f, "preemph_coeff out of [0,1]");
  VB_CHECK(opts->window_type >= 0 && opts->window_type <= 4, "invalid window type %d", opts->window_type);
  const int32_t shift = (int32_t)(opts->samp_freq * 0.001 * opts->frame_shift_ms);  // feature-window.h:92-97
  const int32_t L = (int32_t)(opts->samp_freq * 0.001 * opts->frame_length_ms);
  int np = 1;
  while (np < L) np <<= 1;
  VB_CHECK(L >= 2 && shift >= 1 && np >= 128 && np <= 2048,
           "window %d / shift %d samples (padded %d) outside the supported range", L, shift, np);
  VB_TRY(check_device(device));
  DeviceGuard g(device);
  std::unique_ptr<vbgpu_mfcc_s, decltype(&vbgpu_mfcc_destroy)> h(new vbgpu_mfcc_s, vbgpu_mfcc_destroy);
  h->opts = *opts;
  h->device = device;
  h->shift = shift;
  h->L = L;
  h->npad = np;
  h->log_energy_floor = opts->energy_floor > 0.0f ? logf(opts->energy_floor) : 0.0f;
  h->warps.assign(1, 1.0f);
  VB_TRY(h->stream.create());
  VB_TRY(mfcc_build_tables(h.get()));
  *out = h.release();
  return 0;
}

int vbgpu_mfcc_destroy(vbgpu_mfcc_t h) {
  if (!h) return 0;
  DeviceGuard g(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  delete h;
  return 0;
}

// Columns of the handle's output: num_ceps for MFCC; num_bins (+1 with use_energy) for a filterbank handle.
static inline int32_t feat_dim_of(vbgpu_mfcc_t h) {
  return h->fbank ? h->opts.num_bins + (h->opts.use_energy ? 1 : 0) : h->opts.num_ceps;
}

int vbgpu_mfcc_dim(vbgpu_mfcc_t h) { return h ? feat_dim_of(h) : fail(VBGPU_ERR_INVALID, "null handle"); }

int vbgpu_fbank_create(const vbgpu_mfcc_opts *opts, int32_t use_log_fbank, int32_t use_power, int device, vbgpu_mfcc_t *out) {
  VB_CHECK(opts && out, "null argument");
  vbgpu_mfcc_opts o = *opts;
  o.num_ceps = o.num_bins < 1 ? 1 : o.num_bins;  // unused by the filterbank tail; keeps the shared checks meaningful
  VB_TRY(vbgpu_mfcc_create(&o, device, out));
  (*out)->fbank = 1;
  (*out)->use_log_fbank = use_log_fbank != 0;
  (*out)->use_power = use_power != 0;
  return 0;
}

int vbgpu_plp_create(const vbgpu_mfcc_opts *opts, int32_t lpc_order, float compress_factor, float cepstral_scale, int device,
                     vbgpu_mfcc_t *out) {
  VB_CHECK(opts && out, "null argument");
  VB_CHECK(lpc_order >= 1 && lpc_order <= 30, "lpc_order %d not in [1,30]", lpc_order);
  VB_CHECK(opts->num_ceps <= lpc_order + 1, "num_ceps %d > lpc_order + 1 (feature-plp.cc:126)", opts->num_ceps);
  VB_CHECK(opts->num_bins <= 30, "num_bins %d > 30 for PLP", opts->num_bins);
  VB_TRY(vbgpu_mfcc_create(opts, device, out));
  DeviceGuard g(device);
  std::unique_ptr<vbgpu_mfcc_s, decltype(&vbgpu_mfcc_destroy)> h(*out, vbgpu_mfcc_destroy);
  *out = nullptr;
  h->plp = 1;
  h->lpc_order = lpc_order;
  h->compress_factor = compress_factor;
  h->cepstral_scale = cepstral_scale;
  VB_TRY(mfcc_build_tables(h.get()));  // adds the PLP tables
  *out = h.release();
  return 0;
}


int64_t vbgpu_mfcc_num_frames(vbgpu_mfcc_t h, int64_t n_samples) {
  if (!h) return fail(VBGPU_ERR_INVALID, "null handle");
  return num_frames_of(h, n_samples);
}

int64_t vbgpu_mfcc_frame_offsets(vbgpu_mfcc_t h, const int64_t *sample_offsets, int32_t n_utts, int64_t *frame_offsets) {
  if (!h || !sample_offsets || !frame_offsets || n_utts < 0) return fail(VBGPU_ERR_INVALID, "bad argument");
  frame_offsets[0] = 0;
  for (int32_t u = 0; u < n_utts; u++) {
    const int64_t n = sample_offsets[u + 1] - sample_offsets[u];
    if (n < 0) return fail(VBGPU_ERR_INVALID, "sample_offsets not monotone at utterance %d", u);
    frame_offsets[u + 1] = frame_offsets[u] + num_frames_of(h, n);
  }
  return frame_offsets[n_utts];
}

static int mfcc_compute_host(vbgpu_mfcc_t h, const void *wave, bool is_f32, const int64_t *sample_offsets,
                             int32_t n_utts, const float *vtln_warp, float *out, int32_t out_stride) {
  VB_CHECK(h && sample_offsets && n_utts >= 0, "bad argument");
  VB_CHECK(out_stride >= feat_dim_of(h), "out_stride %d < feature dim %d", out_stride, feat_dim_of(h));
  if (n_utts == 0) return 0;
  VB_CHECK(sample_offsets[0] == 0, "sample_offsets[0] must be 0");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  VB_TRY(mfcc_prepare(h, sample_offsets, n_utts, vtln_warp, s));
  const int64_t T = h->layout.total_frames, ns = sample_offsets[n_utts];
  if (T == 0) return 0;
  VB_CHECK(wave && out, "null buffer");
  const size_t in_bytes = (size_t)ns * (is_f32 ? 4 : 2), out_bytes = (size_t)T * out_stride * 4;
  VB_TRY(h->d_pcm.reserve(in_bytes));
  VB_TRY(h->d_out.reserve(out_bytes));
  VB_TRY(h2d(h->d_pcm.p, wave, in_bytes, s));
  VB_TRY(mfcc_launch(h, h->d_pcm.p, is_f32, h->d_out.as<float>(), out_stride, s));
  VB_TRY(d2h(out, h->d_out.p, out_bytes, s));
  VB_CUDA(cudaStreamSynchronize(s));
  return 0;
}

int vbgpu_mfcc_compute_i16(vbgpu_mfcc_t h, const int16_t *pcm, const int64_t *sample_offsets, int32_t n_utts,
                           const float *vtln_warp, float *out, int32_t out_stride) {
  return mfcc_compute_host(h, pcm, false, sample_offsets, n_utts, vtln_warp, out, out_stride);
}

int vbgpu_mfcc_compute_f32(vbgpu_mfcc_t h, const float *wave, const int64_t *sample_offsets, int32_t n_utts,
                           const float *vtln_warp, float *out, int32_t out_stride) {
  return mfcc_compute_host(h, wave, true, sample_offsets, n_utts, vtln_warp, out, out_stride);
}

int vbgpu_mfcc_compute_dev(vbgpu_mfcc_t h, const void *d_pcm, int32_t is_f32, const int64_t *sample_offsets,
                           int32_t n_utts, const float *vtln_warp, float *d_out, int32_t out_stride, void *stream) {
  VB_CHECK(h && sample_offsets && n_utts >= 0, "bad argument");
  VB_CHECK(out_stride >= feat_dim_of(h), "out_stride %d < feature dim %d", out_stride, feat_dim_of(h));
  if (n_utts == 0) return 0;
  DeviceGuard g(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  VB_TRY(h->order.enter(s));
  VB_TRY(mfcc_prepare(h, sample_offsets, n_utts, vtln_warp, s));
  if (h->layout.total_frames == 0) return 0;
  VB_CHECK(d_pcm && d_out, "null buffer");
  VB_TRY(mfcc_launch(h, d_pcm, is_f32 != 0, d_out, out_stride, s));
  return h->order.leave(s);
}

// ================================================================================================================
// CMVN + feature pipeline
// ================================================================================================================
void vbgpu_feat_opts_default(vbgpu_feat_opts *o) {
  if (!o) return;
  *o = vbgpu_feat_opts{1, 0, 0, 2, 2, 3, 3};
}

int vbgpu_feat_create(const vbgpu_feat_opts *opts, int32_t in_dim, const float *transform, int32_t rows, int32_t cols,
                      int device, vbgpu_feat_t *out) {
  VB_CHECK(opts && out, "null argument");
  *out = nullptr;
  VB_CHECK(in_dim >= 1 && in_dim <= 128, "in_dim %d out of range", in_dim);
  VB_CHECK(opts->mode == 0 || opts->mode == 1, "mode must be 0 (delta) or 1 (lda)");
  VB_CHECK(!opts->norm_vars || opts->norm_means,
           "norm_vars without norm_means is rejected by apply-cmvn (apply-cmvn.cpp:63-65)");
  const int K = in_dim * (opts->splice_left + opts->splice_right + 1);
  if (opts->mode == 0) {
    VB_CHECK(!transform, "delta mode takes no global transform");
    VB_CHECK(opts->delta_order >= 0 && opts->delta_order <= 4 && opts->delta_window >= 1 && opts->delta_window <= 8,
             "delta order %d / window %d unsupported", opts->delta_order, opts->delta_window);
  } else {
    VB_CHECK(opts->splice_left >= 0 && opts->splice_right >= 0 && opts->splice_left <= 16 && opts->splice_right <= 16,
             "splice context out of range");
    VB_CHECK(transform, "lda mode needs the global transform (final.mat)");
    VB_CHECK(cols == K || cols == K + 1, "transform has %d columns, spliced dim is %d (transform-feats.cpp:108-114)", cols,
             K);
    VB_CHECK(rows >= 1 && rows <= 256, "transform rows %d out of range", rows);
  }
  VB_TRY(check_device(device));
  DeviceGuard g(device);
  std::unique_ptr<vbgpu_feat_s, decltype(&vbgpu_feat_destroy)> h(new vbgpu_feat_s, vbgpu_feat_destroy);
  h->opts = *opts;
  h->device = device;
  h->in_dim = in_dim;
  VB_TRY(h->stream.create());
  if (opts->mode == 0) {
    // DeltaFeatures ctor, feature-functions.cc:54-86; rows centred in a table of pitch 2*halo+1
    const int order = opts->delta_order, window = opts->delta_window;
    h->halo = order * window;
    const int pitch = 2 * h->halo + 1;
    std::vector<std::vector<float>> sc(order + 1);
    sc[0].assign(1, 1.0f);
    for (int i = 1; i <= order; i++) {
      const std::vector<float> &prev = sc[i - 1];
      std::vector<float> &cur = sc[i];
      const int prev_off = ((int)prev.size() - 1) / 2, cur_off = prev_off + window;
      cur.assign(prev.size() + 2 * window, 0.0f);
      float normalizer = 0.0f;
      for (int j = -window; j <= window; j++) {
        normalizer += j * j;
        for (int k = -prev_off; k <= prev_off; k++) cur[j + k + cur_off] += (float)j * prev[k + prev_off];
      }
      for (float &v : cur) v *= (float)(1.0 / normalizer);
    }
    h->h_delta_scales.assign((size_t)(order + 1) * pitch, 0.0f);
    for (int i = 0; i <= order; i++) {
      const int mo = ((int)sc[i].size() - 1) / 2;
      for (int j = -mo; j <= mo; j++) h->h_delta_scales[(size_t)i * pitch + h->halo + j] = sc[i][j + mo];
    }
    h->mid_dim = in_dim * (order + 1);
    h->out_dim = h->mid_dim;
    VB_TRY(h->d_delta_scales.upload(h->h_delta_scales.data(), h->h_delta_scales.size() * 4));
  } else {
    h->halo = std::max(opts->splice_left, opts->splice_right);
    h->t_rows = rows;
    h->t_cols = cols;
    h->mid_dim = rows;
    h->out_dim = rows;
    VB_TRY(h->d_transform.upload(transform, (size_t)rows * cols * 4));
  }
  *out = h.release();
  return 0;
}

int vbgpu_feat_destroy(vbgpu_feat_t h) {
  if (!h) return 0;
  DeviceGuard g(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  delete h;
  return 0;
}

int vbgpu_feat_out_dim(vbgpu_feat_t h) { return h ? h->out_dim : fail(VBGPU_ERR_INVALID, "null handle"); }

static int check_spk(const int32_t *utt2spk, int32_t n_utts, int32_t n_spk) {
  if (!utt2spk) {
    VB_CHECK(n_spk == n_utts, "utt2spk is null but n_spk %d != n_utts %d", n_spk, n_utts);
    return 0;
  }
  for (int32_t u = 0; u < n_utts; u++)
    VB_CHECK(utt2spk[u] >= 0 && utt2spk[u] < n_spk, "utt2spk[%d]=%d out of [0,%d)", u, utt2spk[u], n_spk);
  return 0;
}

int vbgpu_cmvn_stats(vbgpu_feat_t h, const float *feats, int32_t stride, const int64_t *frame_offsets, int32_t n_utts,
                     const int32_t *utt2spk, int32_t n_spk, double *stats) {
  VB_CHECK(h && frame_offsets && stats && n_utts >= 0 && n_spk >= 0, "bad argument");
  VB_CHECK(stride >= h->in_dim, "stride %d < dim %d", stride, h->in_dim);
  VB_TRY(check_spk(utt2spk, n_utts, n_spk));
  if (n_utts == 0) return 0;
  VB_CHECK(frame_offsets[0] == 0, "frame_offsets[0] must be 0");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  VB_TRY(h->layout.update(nullptr, frame_offsets, n_utts, utt2spk, nullptr, s));
  const int64_t T = h->layout.total_frames;
  if (T == 0) return 0;
  VB_CHECK(feats, "null feats");
  const size_t nst = (size_t)n_spk * 2 * (h->in_dim + 1);
  VB_TRY(h->d_in.reserve((size_t)T * stride * 4));
  VB_TRY(h->d_stats.reserve(nst * 8));
  VB_TRY(h2d(h->d_in.p, feats, (size_t)T * stride * 4, s));
  VB_CUDA(cudaMemsetAsync(h->d_stats.p, 0, nst * 8, s));
  VB_TRY(feat_launch_stats(h, h->d_in.as<float>(), stride, h->d_stats.as<double>(), n_spk, s));
  std::vector<double> tmp(nst);
  VB_TRY(d2h(tmp.data(), h->d_stats.p, nst * 8, s));
  VB_CUDA(cudaStreamSynchronize(s));
  for (size_t i = 0; i < nst; i++) stats[i] += tmp[i];
  return 0;
}

// Shared by vbgpu_feat_run and the pipelines: stats (device) -> norm table; returns NUMERIC error if a speaker has
// count < 1 (cmvn.cc:80-82) — checked only when `check` (synchronises).
static int feat_norm_from_stats(vbgpu_feat_t h, const double *d_stats, int32_t n_spk, bool check, cudaStream_t s) {
  if (!(h->opts.norm_means || h->opts.norm_vars)) return 0;
  VB_TRY(feat_compute_norm(h, d_stats, n_spk, s));
  if (check) {
    int32_t bad = 0;
    const size_t nfloats = (size_t)n_spk * 2 * h->in_dim;
    VB_CUDA(cudaMemcpyAsync(&bad, h->d_norm.as<float>() + nfloats, 4, cudaMemcpyDeviceToHost, s));
    VB_CUDA(cudaStreamSynchronize(s));
    if (bad) return fail(VBGPU_ERR_NUMERIC, "insufficient or degenerate CMVN stats for %d speaker(s) (count < 1 or NaN)", bad);
  }
  return 0;
}

static int check_fmllr(vbgpu_feat_t h, const float *fmllr, int32_t fmllr_cols) {
  if (!fmllr) return 0;
  VB_CHECK(fmllr_cols == h->mid_dim || fmllr_cols == h->mid_dim + 1,
           "fMLLR matrix has %d columns, feature dim is %d (transform-feats.cpp:108-114)", fmllr_cols, h->mid_dim);
  return 0;
}

static int check_feat_run(vbgpu_feat_t h, int32_t in_stride, const int64_t *frame_offsets, int32_t n_utts,
                          const int32_t *utt2spk, int32_t n_spk, const double *cmvn_stats, const float *fmllr,
                          int32_t fmllr_cols, int32_t out_stride) {
  VB_CHECK(h && frame_offsets && n_utts >= 0 && n_spk >= 0, "bad argument");
  VB_CHECK(in_stride >= h->in_dim, "in_stride %d < dim %d", in_stride, h->in_dim);
  VB_CHECK(out_stride >= h->out_dim, "out_stride %d < out dim %d", out_stride, h->out_dim);
  VB_CHECK(!(h->opts.norm_means || h->opts.norm_vars) || cmvn_stats, "cmvn_stats is null but normalisation is requested");
  VB_TRY(check_spk(utt2spk, n_utts, n_spk));
  VB_TRY(check_fmllr(h, fmllr, fmllr_cols));
  if (n_utts > 0) VB_CHECK(frame_offsets[0] == 0, "frame_offsets[0] must be 0");
  return 0;
}

// Shared by vbgpu_feat_run and vbgpu_feat_run_dev once the layout is on the device: host CMVN statistics -> norm table,
// then the feature kernel from d_in to d_out, on stream s.
static int feat_run_device(vbgpu_feat_t h, const float *d_in, int32_t in_stride, int32_t n_spk, const double *cmvn_stats,
                           bool check_stats, const float *d_fmllr, int32_t fmllr_cols, float *d_out, int32_t out_stride,
                           cudaStream_t s) {
  if (h->opts.norm_means || h->opts.norm_vars) {
    const size_t nst = (size_t)n_spk * 2 * (h->in_dim + 1);
    VB_TRY(h->d_stats.reserve(nst * 8));
    VB_TRY(h2d(h->d_stats.p, cmvn_stats, nst * 8, s));
    VB_TRY(feat_norm_from_stats(h, h->d_stats.as<double>(), n_spk, check_stats, s));
  }
  return feat_launch(h, d_in, in_stride, d_fmllr, fmllr_cols, d_out, out_stride, s);
}

int vbgpu_feat_run(vbgpu_feat_t h, const float *feats, int32_t in_stride, const int64_t *frame_offsets, int32_t n_utts,
                   const int32_t *utt2spk, int32_t n_spk, const double *cmvn_stats, const float *fmllr,
                   int32_t fmllr_cols, float *out, int32_t out_stride) {
  VB_TRY(check_feat_run(h, in_stride, frame_offsets, n_utts, utt2spk, n_spk, cmvn_stats, fmllr, fmllr_cols, out_stride));
  if (n_utts == 0) return 0;
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  VB_TRY(h->layout.update(nullptr, frame_offsets, n_utts, utt2spk, nullptr, s));
  const int64_t T = h->layout.total_frames;
  if (T == 0) return 0;
  VB_CHECK(feats && out, "null buffer");
  VB_TRY(h->d_in.reserve((size_t)T * in_stride * 4));
  VB_TRY(h->d_out.reserve((size_t)T * out_stride * 4));
  VB_TRY(h2d(h->d_in.p, feats, (size_t)T * in_stride * 4, s));
  const float *d_fm = nullptr;
  if (fmllr) {
    const size_t nb = (size_t)n_spk * h->out_dim * fmllr_cols * 4;
    VB_TRY(h->d_fmllr.reserve(nb));
    VB_TRY(h2d(h->d_fmllr.p, fmllr, nb, s));
    d_fm = h->d_fmllr.as<float>();
  }
  VB_TRY(feat_run_device(h, h->d_in.as<float>(), in_stride, n_spk, cmvn_stats, true, d_fm, fmllr_cols,
                         h->d_out.as<float>(), out_stride, s));
  VB_TRY(d2h(out, h->d_out.p, (size_t)T * out_stride * 4, s));
  VB_CUDA(cudaStreamSynchronize(s));
  return 0;
}

int vbgpu_feat_run_dev(vbgpu_feat_t h, const float *d_feats, int32_t in_stride, const int64_t *frame_offsets,
                       int32_t n_utts, const int32_t *utt2spk, int32_t n_spk, const double *cmvn_stats,
                       const float *d_fmllr, int32_t fmllr_cols, float *d_out, int32_t out_stride, void *stream) {
  VB_TRY(check_feat_run(h, in_stride, frame_offsets, n_utts, utt2spk, n_spk, cmvn_stats, d_fmllr, fmllr_cols,
                        out_stride));
  if (n_utts == 0 || frame_offsets[n_utts] == 0) return 0;
  VB_CHECK(d_feats && d_out, "null buffer");
  if (h->opts.norm_means || h->opts.norm_vars) {
    // the statistics are on the host: reject what cmvn_norm_kernel would flag (count < 1, cmvn.cc:80-82) without a
    // round trip, so that the call stays asynchronous
    const int32_t w = 2 * (h->in_dim + 1);
    for (int32_t k = 0; k < n_spk; k++) {
      const double *st = cmvn_stats + (size_t)k * w;
      bool ok = st[h->in_dim] >= 1.0;
      for (int32_t i = 0; i < w && ok; i++) ok = std::isfinite(st[i]);
      if (!ok) return fail(VBGPU_ERR_NUMERIC, "insufficient or degenerate CMVN stats for speaker %d (count < 1 or NaN)", k);
    }
  }
  DeviceGuard g(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  VB_TRY(h->order.enter(s));  // batch layout, statistics and norm table of the handle
  VB_TRY(h->layout.update(nullptr, frame_offsets, n_utts, utt2spk, nullptr, s));
  VB_TRY(feat_run_device(h, d_feats, in_stride, n_spk, cmvn_stats, false, d_fmllr, fmllr_cols, d_out, out_stride, s));
  return h->order.leave(s);
}

// ================================================================================================================
// Model + scoring
// ================================================================================================================
static int pad_dim(int D) {
  const int opts[] = {16, 24, 32, 40, 48, 64};
  for (int v : opts)
    if (D <= v) return v;
  return (D + 3) / 4 * 4;
}

int vbgpu_gmm_create(int32_t P, int32_t D, const int32_t *pdf_offsets, const float *gconsts, const float *miv,
                     const float *iv, int32_t stride, int device, vbgpu_gmm_t *out) {
  VB_CHECK(out, "null argument");
  *out = nullptr;
  VB_CHECK(pdf_offsets && gconsts && miv && iv, "null model array");
  VB_CHECK(P >= 1 && D >= 1 && stride >= D, "bad model shape: P=%d D=%d stride=%d", P, D, stride);
  VB_CHECK(D <= 64, "feature dimension %d: the scoring kernels are built for D <= 64 (tcgen05: D <= 47)", D);
  VB_CHECK(pdf_offsets[0] == 0, "pdf_offsets[0] must be 0");
  int maxM = 0;
  for (int p = 0; p < P; p++) {
    const int M = pdf_offsets[p + 1] - pdf_offsets[p];
    VB_CHECK(M >= 1, "pdf %d has %d Gaussians", p, M);
    maxM = std::max(maxM, M);
  }
  const int N = pdf_offsets[P];
  for (int i = 0; i < N; i++)  // NaN gconst is fatal in the reference (diag-gmm.cc:137-140); -inf is allowed
    VB_CHECK(!(gconsts[i] != gconsts[i]), "gconst %d is NaN", i);
  VB_TRY(check_device(device));
  DeviceGuard g(device);
  std::unique_ptr<vbgpu_gmm_s, decltype(&vbgpu_gmm_destroy)> h(new vbgpu_gmm_s, vbgpu_gmm_destroy);
  h->device = device;
  h->P = P;
  h->N = N;
  h->D = D;
  h->DP = pad_dim(D);
  h->max_pdf_size = maxM;
  h->h_pdf_offsets.assign(pdf_offsets, pdf_offsets + P + 1);
  VB_TRY(h->stream.create());
  std::vector<float> rows((size_t)N * 2 * h->DP, 0.0f);
  for (int i = 0; i < N; i++)
    for (int d = 0; d < D; d++) {
      rows[(size_t)i * 2 * h->DP + d] = miv[(size_t)i * stride + d];
      rows[(size_t)i * 2 * h->DP + h->DP + d] = -0.5f * iv[(size_t)i * stride + d];  // exact scaling
    }
  VB_TRY(h->d_rows.upload(rows.data(), rows.size() * 4));
  VB_TRY(h->d_gconsts.upload(gconsts, (size_t)N * 4));
  VB_TRY(h->d_pdf_offsets.upload(pdf_offsets, (size_t)(P + 1) * 4));
  VB_TRY(h->d_bad.reserve(8));
  VB_CUDA(cudaMemset(h->d_bad.p, 0, 8));
  VB_TRY(score_tc_prepare(h.get(), gconsts, miv, iv, stride));
  *out = h.release();
  return 0;
}

int vbgpu_gmm_destroy(vbgpu_gmm_t h) {
  if (!h) return 0;
  DeviceGuard g(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  score_tc_release(h);
  delete h;
  return 0;
}

int vbgpu_gmm_num_pdfs(vbgpu_gmm_t h) { return h ? h->P : fail(VBGPU_ERR_INVALID, "null handle"); }
int vbgpu_gmm_num_gauss(vbgpu_gmm_t h) { return h ? h->N : fail(VBGPU_ERR_INVALID, "null handle"); }
int vbgpu_gmm_dim(vbgpu_gmm_t h) { return h ? h->D : fail(VBGPU_ERR_INVALID, "null handle"); }

int vbgpu_gmm_set_gconsts(vbgpu_gmm_t h, const float *gconsts) {
  VB_CHECK(h && gconsts, "null argument");
  for (int i = 0; i < h->N; i++) VB_CHECK(!(gconsts[i] != gconsts[i]), "gconst %d is NaN", i);
  DeviceGuard g(h->device);
  VB_CUDA(cudaStreamSynchronize(h->stream));
  VB_CUDA(cudaMemcpy(h->d_gconsts.p, gconsts, (size_t)h->N * 4, cudaMemcpyHostToDevice));
  return score_tc_update_gconsts(h, gconsts);
}

int vbgpu_gmm_set_kernel(vbgpu_gmm_t h, int32_t kind) {
  VB_CHECK(h, "null handle");
  VB_CHECK(kind >= 0 && kind <= 2, "kernel kind must be 0, 1 or 2");
  VB_CHECK(kind != 2 || score_tc_available(h), "tensor-core scorer unavailable for this model (D=%d)", h->D);
  h->kernel = kind;
  return 0;
}

static bool uses_tc(vbgpu_gmm_t h) { return h->kernel == 2 || (h->kernel == 0 && score_tc_available(h)); }
// Columns of the natively laid out score matrix (device column order): the tensor-core kernel's, or P (identity).
static int32_t native_cols(vbgpu_gmm_t h) { return uses_tc(h) ? score_tc_num_cols(h) : h->P; }

// Message of a host scoring form whose call produced NaN/Inf log-likelihoods.
static const char kBadLoglikes[] = "%llu NaN/Inf log-likelihoods (overflow or invalid variances/features?)";

// native: d_ll in device column order (see vbgpu_gmm_score_cols_dev), else in the model's pdf order.
static int score_dispatch(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, float *d_ll,
                          int32_t ll_stride, bool native, unsigned long long *bad, cudaStream_t s) {
  VB_TRY(h->order.enter(s));  // the handle's scratch (row flags, gather scratch) may still be in use on another stream
  VB_TRY(uses_tc(h) ? score_tc_launch(h, d_feats, T, stride, d_ll, ll_stride, native ? 1 : 0, bad, s)
                    : score_simt_launch(h, d_feats, T, stride, d_ll, ll_stride, bad, s));
  return h->order.leave(s);
}

int vbgpu_gmm_score_dev(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, float *d_ll, int32_t ll_stride,
                        void *stream) {
  VB_CHECK(h && T >= 0, "bad argument");
  VB_CHECK(stride >= h->D && ll_stride >= h->P, "stride %d < D %d or ll_stride %d < P %d", stride, h->D, ll_stride, h->P);
  if (T == 0) return 0;
  VB_CHECK(d_feats && d_ll, "null buffer");
  DeviceGuard g(h->device);
  return score_dispatch(h, d_feats, T, stride, d_ll, ll_stride, false, h->d_bad.as<unsigned long long>(),
                        static_cast<cudaStream_t>(stream));
}

int vbgpu_gmm_num_cols(vbgpu_gmm_t h) { return h ? native_cols(h) : fail(VBGPU_ERR_INVALID, "null handle"); }

int vbgpu_gmm_col_of_pdf(vbgpu_gmm_t h, int32_t *col_of_pdf) {
  VB_CHECK(h && col_of_pdf, "null argument");
  const int32_t *m = uses_tc(h) ? score_tc_col_of_pdf(h) : nullptr;
  for (int p = 0; p < h->P; p++) col_of_pdf[p] = m ? m[p] : p;
  return 0;
}

const char *vbgpu_gmm_plan_note(vbgpu_gmm_t h) { return h ? h->tc_note.c_str() : ""; }

int vbgpu_debug_tc_layout(int32_t P, int32_t D, const int32_t *pdf_offsets, const float *gconsts, const float *miv,
                          const float *iv, int32_t stride, int32_t pair, int32_t *info, uint8_t *image, int64_t image_cap,
                          int32_t *hdr, int32_t hdr_cap, int32_t *grp, int32_t grp_cap, int32_t *col_of_pdf, int32_t *merge,
                          int32_t merge_cap, float *centre, float *s1, float *s2, int32_t *bounds) {
  VB_CHECK(pdf_offsets && gconsts && miv && iv && info, "null argument");
  VB_CHECK(P >= 1 && D >= 1 && stride >= D && pdf_offsets[0] == 0, "bad model shape");
  return score_tc_debug_layout(P, D, pdf_offsets, gconsts, miv, iv, stride, pair, info, image, image_cap, hdr, hdr_cap, grp,
                               grp_cap, col_of_pdf, merge, merge_cap, centre, s1, s2, bounds);
}

int vbgpu_gmm_score_cols_dev(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, float *d_ll,
                             int32_t ll_stride, void *stream) {
  VB_CHECK(h && T >= 0, "bad argument");
  VB_CHECK(stride >= h->D && ll_stride >= native_cols(h), "stride %d < D %d or ll_stride %d < %d columns", stride, h->D,
           ll_stride, native_cols(h));
  if (T == 0) return 0;
  VB_CHECK(d_feats && d_ll, "null buffer");
  DeviceGuard g(h->device);
  return score_dispatch(h, d_feats, T, stride, d_ll, ll_stride, true, h->d_bad.as<unsigned long long>(),
                        static_cast<cudaStream_t>(stream));
}

int vbgpu_gmm_bad_count(vbgpu_gmm_t h, int64_t *count) {
  VB_CHECK(h && count, "null argument");
  DeviceGuard g(h->device);
  VB_CUDA(cudaDeviceSynchronize());
  unsigned long long v = 0;
  VB_CUDA(cudaMemcpy(&v, h->d_bad.p, 8, cudaMemcpyDeviceToHost));
  VB_CUDA(cudaMemset(h->d_bad.p, 0, 8));
  *count = (int64_t)v;
  return 0;
}

int vbgpu_gmm_rescored_frames(vbgpu_gmm_t h, int64_t *count) {
  VB_CHECK(h && count, "null argument");
  DeviceGuard g(h->device);
  return vb::score_tc_rescored(h, count);
}

int vbgpu_gmm_score(vbgpu_gmm_t h, const float *feats, int64_t T, int32_t stride, float *loglikes, int32_t ll_stride) {
  VB_CHECK(h && T >= 0, "bad argument");
  VB_CHECK(stride >= h->D && ll_stride >= h->P, "stride %d < D %d or ll_stride %d < P %d", stride, h->D, ll_stride, h->P);
  if (T == 0) return 0;
  VB_CHECK(feats && loglikes, "null buffer");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  // bounded device footprint: score in slabs of at most ~1 GiB of output
  int64_t slab = (int64_t)(1ull << 30) / ((int64_t)ll_stride * 4);
  slab = std::max<int64_t>(256, slab / 256 * 256);
  slab = std::min(slab, T);
  VB_TRY(h->d_feats.reserve((size_t)slab * stride * 4));
  VB_TRY(h->d_ll.reserve((size_t)slab * ll_stride * 4));
  unsigned long long *bad = nullptr, n_bad = 0;
  VB_TRY(h->count.begin(s, &bad));
  for (int64_t t0 = 0; t0 < T; t0 += slab) {
    const int64_t n = std::min(slab, T - t0);
    VB_TRY(h2d(h->d_feats.p, feats + t0 * stride, (size_t)n * stride * 4, s));
    VB_TRY(score_dispatch(h, h->d_feats.as<float>(), n, stride, h->d_ll.as<float>(), ll_stride, false, bad, s));
    VB_TRY(d2h(loglikes + t0 * ll_stride, h->d_ll.p, (size_t)n * ll_stride * 4, s));
    VB_CUDA(cudaStreamSynchronize(s));
  }
  VB_TRY(h->count.end(s, &n_bad));
  if (n_bad) return fail(VBGPU_ERR_NUMERIC, kBadLoglikes, n_bad);
  return 0;
}

// ================================================================================================================
// Sparse consumers of the score matrix (SURVEY.md §8f n3): per-utterance pdf subsets, (frame, pdf) arcs
// ================================================================================================================
namespace {
struct SparseReq {
  int mode = 0;  // 0 = per-utterance subsets, 1 = arcs
  const int32_t *d_f2u = nullptr, *d_cols = nullptr, *d_frames = nullptr;
  const int64_t *d_fo = nullptr, *d_so = nullptr, *d_oo = nullptr;
  int64_t n = 0;       // arcs
  float *d_out = nullptr;
  // subsets through a host-facing call: where the packed result goes on the host, and what is needed to find the output
  // range of a slab of frames (frames are packed utterance after utterance, so a slab's results are one contiguous range)
  float *h_out = nullptr;
  std::vector<int64_t> h_fo, h_oo;
};
}  // namespace

// Dense scoring in slabs of frames (device column order) + extraction of what the request names.  The slab is sized for
// a few waves of the tensor-core kernel and at most ~2 GiB, so the footprint does not depend on T.
static int score_sparse_dev(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, const SparseReq &rq,
                            unsigned long long *bad, cudaStream_t s) {
  if (T == 0) return 0;
  const int32_t st = (native_cols(h) + 3) / 4 * 4;
  const int64_t wave = 256LL * std::max(1, num_sms(h->device) / 2);
  int64_t slab = (int64_t)(2ull << 30) / ((int64_t)st * 4) / wave * wave;
  slab = std::min(std::max(slab, wave), (T + 255) / 256 * 256);
  VB_TRY(h->d_sp_slab.reserve((size_t)slab * st * 4));
  VB_TRY(h->order.enter(s));
  const bool stream_out = rq.mode == 0 && rq.h_out != nullptr;
  if (stream_out && !h->copy_stream) {
    VB_TRY(h->copy_stream.create());
    for (Event &e : h->sp_done) VB_TRY(e.create());
  }
  // first element of frame t in the packed output
  auto out_pos = [&rq](int64_t t) {
    const size_t u = (size_t)(std::upper_bound(rq.h_fo.begin(), rq.h_fo.end(), t) - rq.h_fo.begin()) - 1;
    if (u + 1 >= rq.h_fo.size()) return rq.h_oo.back();
    const int64_t frames = rq.h_fo[u + 1] - rq.h_fo[u];
    return rq.h_oo[u] + (frames > 0 ? (rq.h_oo[u + 1] - rq.h_oo[u]) / frames * (t - rq.h_fo[u]) : 0);
  };
  // the copy of slab k is issued after the launches of slab k + 1, so that a pageable destination (a copy that holds the
  // host thread) still overlaps with scoring
  auto copy_out = [&](int64_t a, int64_t b, int k) -> int {
    const int64_t p0 = out_pos(a), p1 = out_pos(b);
    if (p1 <= p0) return 0;
    VB_CUDA(cudaStreamWaitEvent(h->copy_stream, h->sp_done[k & 1], 0));
    VB_CUDA(cudaMemcpyAsync(rq.h_out + p0, rq.d_out + p0, (size_t)(p1 - p0) * 4, cudaMemcpyDeviceToHost, h->copy_stream));
    return 0;
  };
  int k = 0;
  int64_t prev0 = 0, prev1 = 0;
  for (int64_t t0 = 0; t0 < T; t0 += slab, k++) {
    const int64_t n = std::min(slab, T - t0);
    VB_TRY(score_dispatch(h, d_feats + t0 * stride, n, stride, h->d_sp_slab.as<float>(), st, true, bad, s));
    if (rq.mode == 0)
      VB_TRY(sparse_subset_launch(h->d_sp_slab.as<float>(), st, t0, t0 + n, rq.d_f2u, rq.d_fo, rq.d_so, rq.d_cols, rq.d_oo,
                                  rq.d_out, s));
    else
      VB_TRY(sparse_gather_launch(h->d_sp_slab.as<float>(), st, t0, t0 + n, rq.d_frames, rq.d_cols, rq.n, rq.d_out, s));
    if (stream_out) {
      VB_CUDA(cudaEventRecord(h->sp_done[k & 1], s));
      if (k > 0) VB_TRY(copy_out(prev0, prev1, k - 1));
      prev0 = t0, prev1 = t0 + n;
    }
  }
  if (stream_out) {
    VB_TRY(copy_out(prev0, prev1, k - 1));
    VB_CUDA(cudaStreamSynchronize(h->copy_stream));
  }
  return h->order.leave(s);
}

// Validates and uploads the description of per-utterance subsets; fills rq (device pointers into the handle's scratch)
// and out_offsets / total.
static int sparse_prepare_subset(vbgpu_gmm_t h, int64_t T, const int64_t *frame_offsets, int32_t n_utts,
                                 const int64_t *subset_offsets, const int32_t *subset_pdfs, int64_t *out_offsets,
                                 int64_t *total, SparseReq *rq, cudaStream_t s) {
  VB_CHECK(frame_offsets && subset_offsets && subset_pdfs && n_utts >= 1, "null / empty subset description");
  VB_CHECK(frame_offsets[0] == 0 && frame_offsets[n_utts] == T && subset_offsets[0] == 0, "offsets must start at 0 and cover T");
  const int64_t n_sub = subset_offsets[n_utts];
  std::vector<int64_t> i64((size_t)3 * (n_utts + 1));
  int64_t *fo = i64.data(), *so = fo + n_utts + 1, *oo = so + n_utts + 1;
  oo[0] = 0;
  for (int32_t u = 0; u < n_utts; u++) {
    VB_CHECK(frame_offsets[u + 1] >= frame_offsets[u] && subset_offsets[u + 1] >= subset_offsets[u], "offsets must not decrease");
    oo[u + 1] = oo[u] + (frame_offsets[u + 1] - frame_offsets[u]) * (subset_offsets[u + 1] - subset_offsets[u]);
  }
  std::memcpy(fo, frame_offsets, (size_t)(n_utts + 1) * 8);
  std::memcpy(so, subset_offsets, (size_t)(n_utts + 1) * 8);
  std::vector<int32_t> cols((size_t)std::max<int64_t>(n_sub, 1));
  const int32_t *map = uses_tc(h) ? score_tc_col_of_pdf(h) : nullptr;
  for (int64_t i = 0; i < n_sub; i++) {
    VB_CHECK(subset_pdfs[i] >= 0 && subset_pdfs[i] < h->P, "pdf id %d out of range", subset_pdfs[i]);
    cols[i] = map ? map[subset_pdfs[i]] : subset_pdfs[i];
  }
  if (out_offsets) std::memcpy(out_offsets, oo, (size_t)(n_utts + 1) * 8);
  *total = oo[n_utts];
  rq->h_fo.assign(fo, fo + n_utts + 1);
  rq->h_oo.assign(oo, oo + n_utts + 1);
  VB_TRY(h->d_sp_i64.reserve(i64.size() * 8));
  VB_TRY(h->d_sp_i32.reserve(cols.size() * 4));
  VB_TRY(h->d_sp_f2u.reserve((size_t)std::max<int64_t>(T, 1) * 4));
  VB_CUDA(cudaStreamSynchronize(s));  // (pageable staging below: the previous call's kernels may still read the scratch)
  VB_CUDA(cudaMemcpyAsync(h->d_sp_i64.p, i64.data(), i64.size() * 8, cudaMemcpyHostToDevice, s));
  VB_CUDA(cudaMemcpyAsync(h->d_sp_i32.p, cols.data(), cols.size() * 4, cudaMemcpyHostToDevice, s));
  VB_CUDA(cudaStreamSynchronize(s));
  rq->mode = 0;
  rq->d_fo = h->d_sp_i64.as<int64_t>();
  rq->d_so = rq->d_fo + n_utts + 1;
  rq->d_oo = rq->d_so + n_utts + 1;
  rq->d_cols = h->d_sp_i32.as<int32_t>();
  rq->d_f2u = h->d_sp_f2u.as<int32_t>();
  launch_fill_frame2utt(rq->d_fo, n_utts, T, h->d_sp_f2u.as<int32_t>(), s);
  VB_CUDA(cudaGetLastError());
  return 0;
}

static int sparse_prepare_gather(vbgpu_gmm_t h, int64_t T, const int32_t *frames, const int32_t *pdfs, int64_t n,
                                 SparseReq *rq, cudaStream_t s) {
  VB_CHECK(n >= 0 && (n == 0 || (frames && pdfs)), "null arc list");
  std::vector<int32_t> cols((size_t)std::max<int64_t>(n, 1));
  const int32_t *map = uses_tc(h) ? score_tc_col_of_pdf(h) : nullptr;
  for (int64_t i = 0; i < n; i++) {
    VB_CHECK(frames[i] >= 0 && frames[i] < T, "arc %lld: frame %d outside [0, %lld)", (long long)i, frames[i], (long long)T);
    VB_CHECK(pdfs[i] >= 0 && pdfs[i] < h->P, "arc %lld: pdf id %d out of range", (long long)i, pdfs[i]);
    cols[i] = map ? map[pdfs[i]] : pdfs[i];
  }
  VB_TRY(h->d_sp_i32.reserve((size_t)std::max<int64_t>(n, 1) * 8));
  VB_CUDA(cudaStreamSynchronize(s));
  int32_t *d = h->d_sp_i32.as<int32_t>();
  if (n) {
    VB_CUDA(cudaMemcpyAsync(d, frames, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    VB_CUDA(cudaMemcpyAsync(d + n, cols.data(), (size_t)n * 4, cudaMemcpyHostToDevice, s));
    VB_CUDA(cudaStreamSynchronize(s));
  }
  rq->mode = 1;
  rq->d_frames = d;
  rq->d_cols = d + n;
  rq->n = n;
  return 0;
}

int vbgpu_gmm_score_subset_dev(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, const int64_t *frame_offsets,
                               int32_t n_utts, const int64_t *subset_offsets, const int32_t *subset_pdfs, float *d_out,
                               int64_t *out_offsets, void *stream) {
  VB_CHECK(h && T >= 0 && stride >= h->D, "bad argument");
  DeviceGuard g(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  SparseReq rq;
  int64_t total = 0;
  VB_TRY(sparse_prepare_subset(h, T, frame_offsets, n_utts, subset_offsets, subset_pdfs, out_offsets, &total, &rq, s));
  if (total == 0) return 0;
  VB_CHECK(d_feats && d_out, "null buffer");
  rq.d_out = d_out;
  return score_sparse_dev(h, d_feats, T, stride, rq, h->d_bad.as<unsigned long long>(), s);
}

int vbgpu_gmm_score_subset(vbgpu_gmm_t h, const float *feats, int64_t T, int32_t stride, const int64_t *frame_offsets,
                           int32_t n_utts, const int64_t *subset_offsets, const int32_t *subset_pdfs, float *out,
                           int64_t *out_offsets) {
  VB_CHECK(h && T >= 0 && stride >= h->D, "bad argument");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  SparseReq rq;
  int64_t total = 0;
  VB_TRY(sparse_prepare_subset(h, T, frame_offsets, n_utts, subset_offsets, subset_pdfs, out_offsets, &total, &rq, s));
  if (total == 0) return 0;
  VB_CHECK(feats && out, "null buffer");
  VB_TRY(h->d_feats.reserve((size_t)T * stride * 4));
  VB_TRY(h->d_sp_out.reserve((size_t)total * 4));
  unsigned long long *bad = nullptr, n_bad = 0;
  VB_TRY(h->count.begin(s, &bad));
  VB_TRY(h2d(h->d_feats.p, feats, (size_t)T * stride * 4, s));
  rq.d_out = h->d_sp_out.as<float>();
  rq.h_out = out;  // results leave slab by slab, behind the scoring of the next slab
  VB_TRY(score_sparse_dev(h, h->d_feats.as<float>(), T, stride, rq, bad, s));
  VB_TRY(h->count.end(s, &n_bad));
  if (n_bad) return fail(VBGPU_ERR_NUMERIC, kBadLoglikes, n_bad);
  return 0;
}

int vbgpu_gmm_score_gather_dev(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, const int32_t *frames,
                               const int32_t *pdfs, int64_t n, float *d_out, void *stream) {
  VB_CHECK(h && T >= 0 && stride >= h->D, "bad argument");
  DeviceGuard g(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  SparseReq rq;
  VB_TRY(sparse_prepare_gather(h, T, frames, pdfs, n, &rq, s));
  if (n == 0) return 0;
  VB_CHECK(d_feats && d_out, "null buffer");
  rq.d_out = d_out;
  return score_sparse_dev(h, d_feats, T, stride, rq, h->d_bad.as<unsigned long long>(), s);
}

int vbgpu_gmm_score_gather(vbgpu_gmm_t h, const float *feats, int64_t T, int32_t stride, const int32_t *frames,
                           const int32_t *pdfs, int64_t n, float *out) {
  VB_CHECK(h && T >= 0 && stride >= h->D, "bad argument");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  SparseReq rq;
  VB_TRY(sparse_prepare_gather(h, T, frames, pdfs, n, &rq, s));
  if (n == 0) return 0;
  VB_CHECK(feats && out, "null buffer");
  VB_TRY(h->d_feats.reserve((size_t)T * stride * 4));
  VB_TRY(h->d_sp_out.reserve((size_t)n * 4));
  unsigned long long *bad = nullptr, n_bad = 0;
  VB_TRY(h->count.begin(s, &bad));
  VB_TRY(h2d(h->d_feats.p, feats, (size_t)T * stride * 4, s));
  rq.d_out = h->d_sp_out.as<float>();
  VB_TRY(score_sparse_dev(h, h->d_feats.as<float>(), T, stride, rq, bad, s));
  VB_TRY(d2h(out, h->d_sp_out.p, (size_t)n * 4, s));
  VB_TRY(h->count.end(s, &n_bad));
  if (n_bad) return fail(VBGPU_ERR_NUMERIC, kBadLoglikes, n_bad);
  return 0;
}

// ================================================================================================================
// Forced alignment (graph layout and kernels in align.cu): subset scoring, then Viterbi + traceback, group by group
// ================================================================================================================
int vbgpu_align_create(int32_t n_utts, const int32_t *state_offsets, const int32_t *start, const float *final_cost,
                       const int64_t *arc_offsets, const int32_t *arc_src, const int32_t *arc_dst, const int32_t *arc_ilabel,
                       const float *arc_weight, const int32_t *tid2pdf, int32_t num_tids, int device, vbgpu_align_t *out) {
  return align_create(n_utts, state_offsets, start, final_cost, arc_offsets, arc_src, arc_dst, arc_ilabel, arc_weight,
                      tid2pdf, num_tids, device, out);
}

int vbgpu_align_destroy(vbgpu_align_t h) {
  if (!h) return 0;
  DeviceGuard g(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  delete h;
  return 0;
}

int vbgpu_align_set_workspace(vbgpu_align_t h, int64_t bytes) {
  VB_CHECK(h, "null handle");
  h->workspace_cap = bytes > 0 ? bytes : kAlignDefaultWorkspace;
  return 0;
}

static int check_align_args(vbgpu_align_t h, vbgpu_gmm_t model, const float *tid_cost, int32_t stride,
                            const int64_t *frame_offsets, int32_t n_utts) {
  VB_CHECK(h && model && frame_offsets, "null argument");
  VB_CHECK(n_utts == h->n_utts, "frame_offsets describe %d utterances, the graphs %d", n_utts, h->n_utts);
  VB_CHECK(model->device == h->device, "model on device %d, graphs on device %d", model->device, h->device);
  VB_CHECK(h->max_pdf < model->P, "tid2pdf names pdf %d, the model has %d", h->max_pdf, model->P);
  VB_CHECK(stride >= model->D, "stride %d < dim %d", stride, model->D);
  VB_CHECK(frame_offsets[0] == 0, "frame_offsets[0] = %lld, not 0", (long long)frame_offsets[0]);
  for (int32_t u = 0; u < n_utts; u++)
    VB_CHECK(frame_offsets[u + 1] >= frame_offsets[u], "frame_offsets not monotone at utterance %d", u);
  if (tid_cost)
    for (int32_t i = 1; i <= h->num_tids; i++)
      VB_CHECK(!std::isnan(tid_cost[i]) && tid_cost[i] != -INFINITY, "tid_cost[%d] is NaN or -inf", i);
  return 0;
}

// Everything behind the argument checks, on device buffers; bad receives the count of non-finite log-likelihoods.
static int align_run(vbgpu_align_t h, vbgpu_gmm_t model, const float *tid_cost, float scale, const float *d_feats,
                     int32_t stride, const int64_t *fo, int32_t *d_ali, int32_t *d_pdf, double *d_tot,
                     unsigned long long *bad, cudaStream_t s) {
  const int32_t n = h->n_utts;
  const int64_t tbb = h->tb_bytes;
  std::vector<AlignCall> calls((size_t)n);
  std::vector<int32_t> group_end;  // utterance after each group
  int64_t tb_max = 0, ll_max = 0, tb_g = 0, ll_g = 0;
  for (int32_t u = 0; u < n; u++) {
    const int64_t T = fo[u + 1] - fo[u], tb = (T + 1) * h->h_S[u] * tbb, ll = T * h->h_nsub[u] * 4;
    if (u > 0 && tb_g + ll_g + tb + ll > h->workspace_cap) group_end.push_back(u), tb_g = ll_g = 0;
    calls[u] = AlignCall{fo[u], T, ll_g / 4, tb_g / tbb};
    tb_g += tb, ll_g += ll;
    tb_max = std::max(tb_max, tb_g), ll_max = std::max(ll_max, ll_g);
  }
  group_end.push_back(n);
  VB_TRY(h->order.enter(s));
  VB_TRY(h->d_tb.reserve((size_t)std::max<int64_t>(tb_max, 16)));
  VB_TRY(h->d_ll.reserve((size_t)std::max<int64_t>(ll_max, 16)));
  VB_TRY(h2d(h->d_calls.p, calls.data(), calls.size() * sizeof(AlignCall), s));
  VB_TRY(align_set_weights(h, tid_cost, s));
  std::vector<int64_t> g_fo, g_so;
  int32_t u0 = 0;
  for (int32_t u1 : group_end) {
    const int32_t k = u1 - u0;
    g_fo.assign((size_t)k + 1, 0);
    g_so.assign((size_t)k + 1, 0);
    int32_t max_S = 1, max_sub = 0;
    for (int32_t i = 0; i < k; i++) {
      g_fo[i + 1] = fo[u0 + i + 1] - fo[u0];
      g_so[i + 1] = h->h_sub_off[u0 + i + 1] - h->h_sub_off[u0];
      max_S = std::max(max_S, h->h_S[u0 + i]);
      max_sub = std::max(max_sub, h->h_nsub[u0 + i]);
    }
    const int64_t Tg = g_fo[k];
    SparseReq rq;
    int64_t total = 0;
    VB_TRY(sparse_prepare_subset(model, Tg, g_fo.data(), k, g_so.data(), h->h_sub_pdfs.data() + h->h_sub_off[u0], nullptr,
                                 &total, &rq, s));
    if (total > 0) {
      rq.d_out = h->d_ll.as<float>();
      VB_TRY(score_sparse_dev(model, d_feats + fo[u0] * stride, Tg, stride, rq, bad, s));
    }
    VB_TRY(align_group_launch(h, u0, k, max_S, max_sub, h->d_ll.as<float>(), scale, h->d_tb.p, d_ali, d_pdf, d_tot, s));
    u0 = u1;
  }
  return h->order.leave(s);
}

int vbgpu_align_dev(vbgpu_align_t h, vbgpu_gmm_t model, const float *tid_cost, float acoustic_scale, const float *d_feats,
                    int32_t stride, const int64_t *frame_offsets, int32_t n_utts, int32_t *d_ali, int32_t *d_pdf_ids,
                    double *d_tot_cost, void *stream) {
  VB_TRY(check_align_args(h, model, tid_cost, stride, frame_offsets, n_utts));
  VB_CHECK(d_tot_cost && (frame_offsets[n_utts] == 0 || (d_feats && d_ali)), "null buffer");
  DeviceGuard g(h->device);
  return align_run(h, model, tid_cost, acoustic_scale, d_feats, stride, frame_offsets, d_ali, d_pdf_ids, d_tot_cost,
                   model->d_bad.as<unsigned long long>(), static_cast<cudaStream_t>(stream));
}

int vbgpu_align(vbgpu_align_t h, vbgpu_gmm_t model, const float *tid_cost, float acoustic_scale, const float *feats,
                int32_t stride, const int64_t *frame_offsets, int32_t n_utts, int32_t *ali, int32_t *pdf_ids,
                double *tot_cost) {
  VB_TRY(check_align_args(h, model, tid_cost, stride, frame_offsets, n_utts));
  const int64_t T = frame_offsets[n_utts];
  VB_CHECK(tot_cost && (T == 0 || (feats && ali)), "null buffer");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  const size_t rows = (size_t)std::max<int64_t>(T, 1);
  VB_TRY(h->d_feats.reserve(rows * stride * 4));
  VB_TRY(h->d_ali.reserve(rows * 4));
  VB_TRY(h->d_pdf.reserve(rows * 4));
  VB_TRY(h->d_tot.reserve((size_t)n_utts * 8));
  unsigned long long *bad = nullptr, n_bad = 0;
  VB_TRY(h->count.begin(s, &bad));
  VB_TRY(h2d(h->d_feats.p, feats, (size_t)T * stride * 4, s));
  VB_TRY(align_run(h, model, tid_cost, acoustic_scale, h->d_feats.as<float>(), stride, frame_offsets, h->d_ali.as<int32_t>(),
                   pdf_ids ? h->d_pdf.as<int32_t>() : nullptr, h->d_tot.as<double>(), bad, s));
  VB_TRY(d2h(ali, h->d_ali.p, (size_t)T * 4, s));
  if (pdf_ids) VB_TRY(d2h(pdf_ids, h->d_pdf.p, (size_t)T * 4, s));
  VB_TRY(d2h(tot_cost, h->d_tot.p, (size_t)n_utts * 8, s));
  VB_TRY(h->count.end(s, &n_bad));
  if (n_bad) return fail(VBGPU_ERR_NUMERIC, kBadLoglikes, n_bad);
  return 0;
}

// ================================================================================================================
// Decoding (graph layout and kernels in decode.cu): dense scoring (feature form), then search + traceback, group by group
// ================================================================================================================
void vbgpu_decoder_opts_default(vbgpu_decoder_opts *o) {
  if (!o) return;
  o->beam = 16.0f;
  o->max_active = INT32_MAX;
  o->max_tokens = 65536;
}

int vbgpu_decoder_create(int32_t num_states, int32_t start, const float *final_cost, int64_t num_arcs,
                         const int32_t *arc_src, const int32_t *arc_dst, const int32_t *arc_ilabel,
                         const int32_t *arc_olabel, const float *arc_weight, const int32_t *tid2pdf, int32_t num_tids,
                         int device, vbgpu_decoder_t *out) {
  return decoder_create(num_states, start, final_cost, num_arcs, arc_src, arc_dst, arc_ilabel, arc_olabel, arc_weight,
                        tid2pdf, num_tids, device, out);
}

int vbgpu_decoder_destroy(vbgpu_decoder_t h) {
  if (!h) return 0;
  DeviceGuard g(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  delete h;
  return 0;
}

int vbgpu_decoder_set_workspace(vbgpu_decoder_t h, int64_t bytes) {
  VB_CHECK(h, "null handle");
  h->workspace_cap = bytes > 0 ? bytes : kDecodeDefaultWorkspace;
  return 0;
}

static int check_decode_args(vbgpu_decoder_t h, vbgpu_gmm_t model, const vbgpu_decoder_opts *o,
                             const int64_t *frame_offsets, int32_t n_utts, int32_t max_words) {
  VB_CHECK(h && model && o && frame_offsets, "null argument");
  VB_CHECK(n_utts >= 0, "n_utts %d is negative", n_utts);
  VB_CHECK(model->device == h->device, "model on device %d, graph on device %d", model->device, h->device);
  VB_CHECK(h->max_pdf < model->P, "tid2pdf names pdf %d, the model has %d", h->max_pdf, model->P);
  VB_CHECK(o->beam > 0.0f, "beam %g must be > 0", (double)o->beam);
  VB_CHECK(o->max_active >= 1, "max_active %d must be >= 1", o->max_active);
  VB_CHECK(o->max_tokens >= 1, "max_tokens %d must be >= 1", o->max_tokens);
  VB_CHECK(max_words >= 0, "max_words %d is negative", max_words);
  VB_CHECK(frame_offsets[0] == 0, "frame_offsets[0] = %lld, not 0", (long long)frame_offsets[0]);
  for (int32_t u = 0; u < n_utts; u++)
    VB_CHECK(frame_offsets[u + 1] >= frame_offsets[u], "frame_offsets not monotone at utterance %d", u);
  return 0;
}

// Everything behind the argument checks, on device buffers.  feats: d_in is [T x in_stride] features, scored group by
// group into the handle's scratch (bad receives the scorer's count); else d_in is the [T x in_stride] log-likelihoods
// in device column order (bad receives their non-finite entries).
// lo / lat (both or neither): the lattice form, whose lattice store each utterance's workspace also holds.
static int decode_run(vbgpu_decoder_t h, vbgpu_gmm_t model, const vbgpu_decoder_opts *o, float scale, bool feats,
                      const float *d_in, int32_t in_stride, const int64_t *fo, int32_t n, int32_t *d_ali, int32_t *d_pdf,
                      int32_t *d_words, int32_t max_words, int32_t *d_nw, double *d_tot, int32_t *d_status,
                      unsigned long long *bad, cudaStream_t s, const vbgpu_lattice_opts *lo = nullptr,
                      const vbgpu_lattice_out *lat = nullptr) {
  if (n == 0) return 0;
  const int32_t cap = std::min(o->max_tokens, h->S), cap2 = std::min(cap, o->max_active);
  const float *d_feats = feats ? d_in : nullptr, *d_ll = feats ? nullptr : d_in;
  const int32_t stride = in_stride, ll_stride = feats ? native_cols(model) : in_stride;
  std::vector<DecodeCall> calls((size_t)n);
  std::vector<int32_t> group_end;
  int64_t ws_max = 0, ll_max = 0, ws_g = 0, ll_g = 0;
  for (int32_t u = 0; u < n; u++) {
    const int64_t T = fo[u + 1] - fo[u], ws1 = (decode_ws_bytes(h->S, cap, cap2, h->n_lvls, T) + 255) & ~int64_t(255);
    const int32_t NT = lo ? (int32_t)((T + 1) * lo->arena_tokens) : 0, NL = lo ? (int32_t)((T + 1) * lo->arena_links) : 0;
    const int64_t ws = ws1 + (lo ? (lattice_arena_bytes(NT, NL, cap, cap2, T) + 255) & ~int64_t(255) : 0);
    const int64_t ll = feats ? T * ll_stride * 4 : 0;
    if (u > 0 && ws_g + ll_g + ws + ll > h->workspace_cap) group_end.push_back(u), ws_g = ll_g = 0;
    calls[u] = DecodeCall{fo[u], T, feats ? ll_g / ((int64_t)ll_stride * 4) : fo[u], ws_g, ws_g + ws1, NT, NL};
    ws_g += ws, ll_g += ll;
    ws_max = std::max(ws_max, ws_g), ll_max = std::max(ll_max, ll_g);
  }
  group_end.push_back(n);
  VB_TRY(h->order.enter(s));
  VB_TRY(h->d_ws.reserve((size_t)ws_max));
  if (feats) VB_TRY(h->d_ll.reserve((size_t)std::max<int64_t>(ll_max, 16)));
  VB_TRY(h->d_best.reserve((size_t)n * 4));
  VB_TRY(h->d_calls.reserve(calls.size() * sizeof(DecodeCall)));
  VB_TRY(h2d(h->d_calls.p, calls.data(), calls.size() * sizeof(DecodeCall), s));
  const int32_t *cop = uses_tc(model) ? score_tc_col_of_pdf_dev(model) : nullptr;
  VB_TRY(decoder_set_cols(h, cop, s));
  if (!feats) VB_TRY(decoder_count_bad(d_ll, ll_stride, fo[n], cop, model->P, bad, s));
  DecodeArgs a{};
  a.calls = h->d_calls.as<DecodeCall>();
  a.ws = h->d_ws.as<unsigned char>();
  a.e_off = h->d_e_off.as<int32_t>(), a.x_off = h->d_x_off.as<int32_t>(), a.lvl = h->d_lvl.as<int32_t>();
  a.e_arcs = h->d_e_arcs.as<int4>(), a.x_arcs = h->d_x_arcs.as<int4>();
  a.finals = h->d_final.as<float>();
  a.ll = feats ? h->d_ll.as<float>() : d_ll;
  a.ll_stride = ll_stride;
  a.scale = scale, a.beam = o->beam;
  a.max_active = o->max_active, a.S = h->S, a.start = h->start, a.n_lvls = h->n_lvls, a.cap = cap, a.cap2 = cap2;
  a.max_words = max_words;
  a.best = h->d_best.as<int32_t>(), a.status = d_status, a.ali = d_ali, a.pdf_ids = d_pdf, a.words = d_words;
  a.num_words = d_nw, a.tot_cost = d_tot;
  if (lo) {
    a.lattice_beam = lo->lattice_beam, a.max_states = lo->max_states, a.max_arcs = lo->max_arcs;
    a.ilabel = h->d_ilabel.as<int32_t>(), a.olabel = h->d_olabel.as<int32_t>(), a.weight = h->d_weight.as<float>();
    a.lat = *lat;
  }
  int32_t u0 = 0;
  for (int32_t u1 : group_end) {
    if (feats && fo[u1] > fo[u0])
      VB_TRY(score_dispatch(model, d_feats + fo[u0] * stride, fo[u1] - fo[u0], stride, h->d_ll.as<float>(), ll_stride,
                            true, bad, s));
    VB_TRY(decoder_search_launch(a, u0, u1 - u0, lo != nullptr, s));
    VB_TRY(decoder_traceback_launch(h, a, u0, u1 - u0, s));
    if (lo) VB_TRY(decoder_lattice_launch(a, u0, u1 - u0, s));
    u0 = u1;
  }
  return h->order.leave(s);
}

int vbgpu_decode_dev(vbgpu_decoder_t h, vbgpu_gmm_t model, const vbgpu_decoder_opts *o, float acoustic_scale,
                     const float *d_feats, int32_t stride, const int64_t *frame_offsets, int32_t n_utts, int32_t *d_ali,
                     int32_t *d_pdf_ids, int32_t *d_words, int32_t max_words, int32_t *d_num_words, double *d_tot_cost,
                     int32_t *d_status, void *stream) {
  VB_TRY(check_decode_args(h, model, o, frame_offsets, n_utts, max_words));
  VB_CHECK(stride >= model->D, "stride %d < dim %d", stride, model->D);
  const int64_t T = n_utts ? frame_offsets[n_utts] : 0;
  VB_CHECK(n_utts == 0 || (d_num_words && d_tot_cost && d_status && (T == 0 || (d_feats && d_ali)) &&
                           (max_words == 0 || d_words)), "null buffer");
  DeviceGuard g(h->device);
  return decode_run(h, model, o, acoustic_scale, true, d_feats, stride, frame_offsets, n_utts, d_ali, d_pdf_ids, d_words, max_words, d_num_words, d_tot_cost,
                    d_status, model->d_bad.as<unsigned long long>(), static_cast<cudaStream_t>(stream));
}

int vbgpu_decode_loglikes_dev(vbgpu_decoder_t h, vbgpu_gmm_t model, const vbgpu_decoder_opts *o, float acoustic_scale,
                              const float *d_loglikes, int32_t ll_stride, const int64_t *frame_offsets, int32_t n_utts,
                              int32_t *d_ali, int32_t *d_pdf_ids, int32_t *d_words, int32_t max_words,
                              int32_t *d_num_words, double *d_tot_cost, int32_t *d_status, void *stream) {
  VB_TRY(check_decode_args(h, model, o, frame_offsets, n_utts, max_words));
  VB_CHECK(ll_stride >= native_cols(model), "ll_stride %d < the model's %d columns", ll_stride, native_cols(model));
  const int64_t T = n_utts ? frame_offsets[n_utts] : 0;
  VB_CHECK(n_utts == 0 || (d_num_words && d_tot_cost && d_status && (T == 0 || (d_loglikes && d_ali)) &&
                           (max_words == 0 || d_words)), "null buffer");
  DeviceGuard g(h->device);
  return decode_run(h, model, o, acoustic_scale, false, d_loglikes, ll_stride, frame_offsets, n_utts, d_ali,
                    d_pdf_ids, d_words, max_words, d_num_words, d_tot_cost, d_status,
                    model->d_bad.as<unsigned long long>(), static_cast<cudaStream_t>(stream));
}

int vbgpu_decode(vbgpu_decoder_t h, vbgpu_gmm_t model, const vbgpu_decoder_opts *o, float acoustic_scale,
                 const float *feats, int32_t stride, const int64_t *frame_offsets, int32_t n_utts, int32_t *ali,
                 int32_t *pdf_ids, int32_t *words, int32_t max_words, int32_t *num_words, double *tot_cost,
                 int32_t *status) {
  VB_TRY(check_decode_args(h, model, o, frame_offsets, n_utts, max_words));
  VB_CHECK(stride >= model->D, "stride %d < dim %d", stride, model->D);
  const int64_t T = n_utts ? frame_offsets[n_utts] : 0;
  VB_CHECK(n_utts == 0 || (num_words && tot_cost && status && (T == 0 || (feats && ali)) && (max_words == 0 || words)),
           "null buffer");
  if (n_utts == 0) return 0;
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  const size_t rows = (size_t)std::max<int64_t>(T, 1), nw = (size_t)n_utts * max_words;
  VB_TRY(h->d_feats.reserve(rows * stride * 4));
  VB_TRY(h->d_ali.reserve(rows * 4));
  VB_TRY(h->d_pdf.reserve(rows * 4));
  VB_TRY(h->d_words.reserve(std::max<size_t>(nw, 1) * 4));
  VB_TRY(h->d_nw.reserve((size_t)n_utts * 4));
  VB_TRY(h->d_tot.reserve((size_t)n_utts * 8));
  VB_TRY(h->d_status.reserve((size_t)n_utts * 4));
  unsigned long long *bad = nullptr, n_bad = 0;
  VB_TRY(h->count.begin(s, &bad));
  VB_TRY(h2d(h->d_feats.p, feats, (size_t)T * stride * 4, s));
  VB_TRY(decode_run(h, model, o, acoustic_scale, true, h->d_feats.as<float>(), stride, frame_offsets, n_utts,
                    h->d_ali.as<int32_t>(), pdf_ids ? h->d_pdf.as<int32_t>() : nullptr, h->d_words.as<int32_t>(),
                    max_words, h->d_nw.as<int32_t>(), h->d_tot.as<double>(), h->d_status.as<int32_t>(), bad, s));
  VB_TRY(d2h(ali, h->d_ali.p, (size_t)T * 4, s));
  if (pdf_ids) VB_TRY(d2h(pdf_ids, h->d_pdf.p, (size_t)T * 4, s));
  if (nw) VB_TRY(d2h(words, h->d_words.p, nw * 4, s));
  VB_TRY(d2h(num_words, h->d_nw.p, (size_t)n_utts * 4, s));
  VB_TRY(d2h(tot_cost, h->d_tot.p, (size_t)n_utts * 8, s));
  VB_TRY(d2h(status, h->d_status.p, (size_t)n_utts * 4, s));
  VB_TRY(h->count.end(s, &n_bad));
  if (n_bad) return fail(VBGPU_ERR_NUMERIC, kBadLoglikes, n_bad);
  return 0;
}

// Lattice generation: decode_run's lattice form (store and kernels in decode.cu)
void vbgpu_lattice_opts_default(vbgpu_lattice_opts *o) {
  if (!o) return;
  o->lattice_beam = 10.0f;
  o->max_states = 131072;
  o->max_arcs = 524288;
  o->arena_tokens = 8192;
  o->arena_links = 24576;
}

static int check_lattice_args(const vbgpu_lattice_opts *lo, const vbgpu_lattice_out *out, const int64_t *fo,
                              int32_t n_utts) {
  VB_CHECK(lo && out, "null argument");
  VB_CHECK(lo->lattice_beam >= 0.0f, "lattice_beam %g must be >= 0", (double)lo->lattice_beam);
  VB_CHECK(lo->max_states >= 0 && lo->max_arcs >= 0, "max_states %d / max_arcs %d is negative", lo->max_states,
           lo->max_arcs);
  VB_CHECK(lo->arena_tokens >= 1 && lo->arena_links >= 1, "arena_tokens %d / arena_links %d must be >= 1",
           lo->arena_tokens, lo->arena_links);
  for (int32_t u = 0; u < n_utts; u++) {
    const int64_t T1 = fo[u + 1] - fo[u] + 1;
    VB_CHECK(T1 * lo->arena_tokens < (1ll << 31) && T1 * lo->arena_links < (1ll << 31),
             "utterance %d: (T + 1) x arena_tokens / arena_links reaches 2^31", u);
  }
  VB_CHECK(n_utts == 0 || (out->num_states && out->num_arcs && out->lattice_status), "null lattice buffer");
  VB_CHECK(n_utts == 0 || lo->max_states == 0 || (out->state_frame && out->state_graph && out->state_final),
           "null lattice state buffer");
  VB_CHECK(n_utts == 0 || lo->max_arcs == 0 || (out->arc_src && out->arc_dst && out->arc_ilabel && out->arc_olabel &&
                                                out->arc_graph_cost && out->arc_ac_cost),
           "null lattice arc buffer");
  return 0;
}

int vbgpu_decode_lattice_dev(vbgpu_decoder_t h, vbgpu_gmm_t model, const vbgpu_decoder_opts *o,
                             const vbgpu_lattice_opts *lo, float acoustic_scale, const float *d_feats, int32_t stride,
                             const int64_t *frame_offsets, int32_t n_utts, int32_t *d_ali, int32_t *d_pdf_ids,
                             int32_t *d_words, int32_t max_words, int32_t *d_num_words, double *d_tot_cost,
                             int32_t *d_status, const vbgpu_lattice_out *out, void *stream) {
  VB_TRY(check_decode_args(h, model, o, frame_offsets, n_utts, max_words));
  VB_TRY(check_lattice_args(lo, out, frame_offsets, n_utts));
  VB_CHECK(stride >= model->D, "stride %d < dim %d", stride, model->D);
  const int64_t T = n_utts ? frame_offsets[n_utts] : 0;
  VB_CHECK(n_utts == 0 || (d_num_words && d_tot_cost && d_status && (T == 0 || (d_feats && d_ali)) &&
                           (max_words == 0 || d_words)), "null buffer");
  DeviceGuard g(h->device);
  return decode_run(h, model, o, acoustic_scale, true, d_feats, stride, frame_offsets, n_utts, d_ali, d_pdf_ids,
                    d_words, max_words, d_num_words, d_tot_cost, d_status, model->d_bad.as<unsigned long long>(),
                    static_cast<cudaStream_t>(stream), lo, out);
}

int vbgpu_decode_lattice_loglikes_dev(vbgpu_decoder_t h, vbgpu_gmm_t model, const vbgpu_decoder_opts *o,
                                      const vbgpu_lattice_opts *lo, float acoustic_scale, const float *d_loglikes,
                                      int32_t ll_stride, const int64_t *frame_offsets, int32_t n_utts, int32_t *d_ali,
                                      int32_t *d_pdf_ids, int32_t *d_words, int32_t max_words, int32_t *d_num_words,
                                      double *d_tot_cost, int32_t *d_status, const vbgpu_lattice_out *out,
                                      void *stream) {
  VB_TRY(check_decode_args(h, model, o, frame_offsets, n_utts, max_words));
  VB_TRY(check_lattice_args(lo, out, frame_offsets, n_utts));
  VB_CHECK(ll_stride >= native_cols(model), "ll_stride %d < the model's %d columns", ll_stride, native_cols(model));
  const int64_t T = n_utts ? frame_offsets[n_utts] : 0;
  VB_CHECK(n_utts == 0 || (d_num_words && d_tot_cost && d_status && (T == 0 || (d_loglikes && d_ali)) &&
                           (max_words == 0 || d_words)), "null buffer");
  DeviceGuard g(h->device);
  return decode_run(h, model, o, acoustic_scale, false, d_loglikes, ll_stride, frame_offsets, n_utts, d_ali,
                    d_pdf_ids, d_words, max_words, d_num_words, d_tot_cost, d_status,
                    model->d_bad.as<unsigned long long>(), static_cast<cudaStream_t>(stream), lo, out);
}

int vbgpu_decode_lattice(vbgpu_decoder_t h, vbgpu_gmm_t model, const vbgpu_decoder_opts *o, const vbgpu_lattice_opts *lo,
                         float acoustic_scale, const float *feats, int32_t stride, const int64_t *frame_offsets,
                         int32_t n_utts, int32_t *ali, int32_t *pdf_ids, int32_t *words, int32_t max_words,
                         int32_t *num_words, double *tot_cost, int32_t *status, const vbgpu_lattice_out *out) {
  VB_TRY(check_decode_args(h, model, o, frame_offsets, n_utts, max_words));
  VB_TRY(check_lattice_args(lo, out, frame_offsets, n_utts));
  VB_CHECK(stride >= model->D, "stride %d < dim %d", stride, model->D);
  const int64_t T = n_utts ? frame_offsets[n_utts] : 0;
  VB_CHECK(n_utts == 0 || (num_words && tot_cost && status && (T == 0 || (feats && ali)) && (max_words == 0 || words)),
           "null buffer");
  if (n_utts == 0) return 0;
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  const size_t rows = (size_t)std::max<int64_t>(T, 1), nw = (size_t)n_utts * max_words;
  const size_t nst = (size_t)n_utts * lo->max_states, nar = (size_t)n_utts * lo->max_arcs;
  VB_TRY(h->d_feats.reserve(rows * stride * 4));
  VB_TRY(h->d_ali.reserve(rows * 4));
  VB_TRY(h->d_pdf.reserve(rows * 4));
  VB_TRY(h->d_words.reserve(std::max<size_t>(nw, 1) * 4));
  VB_TRY(h->d_nw.reserve((size_t)n_utts * 4));
  VB_TRY(h->d_tot.reserve((size_t)n_utts * 8));
  VB_TRY(h->d_status.reserve((size_t)n_utts * 4));
  // staging: 3 state arrays, 6 arc arrays (all 4 bytes), then num_states, num_arcs, lattice_status, arena_peak x 2
  for (int i = 0; i < 9; i++) VB_TRY(h->d_lat[i].reserve(std::max<size_t>(i < 3 ? nst : nar, 1) * 4));
  VB_TRY(h->d_lat_n.reserve((size_t)n_utts * 5 * 4));
  void *host_arr[9] = {out->state_frame, out->state_graph, out->state_final, out->arc_src, out->arc_dst,
                       out->arc_ilabel, out->arc_olabel, out->arc_graph_cost, out->arc_ac_cost};
  int32_t *dn = h->d_lat_n.as<int32_t>();
  vbgpu_lattice_out d{};
  d.state_frame = h->d_lat[0].as<int32_t>(), d.state_graph = h->d_lat[1].as<int32_t>();
  d.state_final = h->d_lat[2].as<float>();
  d.arc_src = h->d_lat[3].as<int32_t>(), d.arc_dst = h->d_lat[4].as<int32_t>();
  d.arc_ilabel = h->d_lat[5].as<int32_t>(), d.arc_olabel = h->d_lat[6].as<int32_t>();
  d.arc_graph_cost = h->d_lat[7].as<float>(), d.arc_ac_cost = h->d_lat[8].as<float>();
  d.num_states = dn, d.num_arcs = dn + n_utts, d.lattice_status = dn + 2 * n_utts;
  d.arena_peak = out->arena_peak ? dn + 3 * n_utts : nullptr;
  unsigned long long *bad = nullptr, n_bad = 0;
  VB_TRY(h->count.begin(s, &bad));
  VB_TRY(h2d(h->d_feats.p, feats, (size_t)T * stride * 4, s));
  VB_TRY(decode_run(h, model, o, acoustic_scale, true, h->d_feats.as<float>(), stride, frame_offsets, n_utts,
                    h->d_ali.as<int32_t>(), pdf_ids ? h->d_pdf.as<int32_t>() : nullptr, h->d_words.as<int32_t>(),
                    max_words, h->d_nw.as<int32_t>(), h->d_tot.as<double>(), h->d_status.as<int32_t>(), bad, s, lo, &d));
  VB_TRY(d2h(ali, h->d_ali.p, (size_t)T * 4, s));
  if (pdf_ids) VB_TRY(d2h(pdf_ids, h->d_pdf.p, (size_t)T * 4, s));
  if (nw) VB_TRY(d2h(words, h->d_words.p, nw * 4, s));
  VB_TRY(d2h(num_words, h->d_nw.p, (size_t)n_utts * 4, s));
  VB_TRY(d2h(tot_cost, h->d_tot.p, (size_t)n_utts * 8, s));
  VB_TRY(d2h(status, h->d_status.p, (size_t)n_utts * 4, s));
  for (int i = 0; i < 9; i++)
    if ((i < 3 ? nst : nar) > 0) VB_TRY(d2h(host_arr[i], h->d_lat[i].p, (i < 3 ? nst : nar) * 4, s));
  VB_TRY(d2h(out->num_states, d.num_states, (size_t)n_utts * 4, s));
  VB_TRY(d2h(out->num_arcs, d.num_arcs, (size_t)n_utts * 4, s));
  VB_TRY(d2h(out->lattice_status, d.lattice_status, (size_t)n_utts * 4, s));
  if (out->arena_peak) VB_TRY(d2h(out->arena_peak, d.arena_peak, (size_t)n_utts * 8, s));
  VB_TRY(h->count.end(s, &n_bad));
  if (n_bad) return fail(VBGPU_ERR_NUMERIC, kBadLoglikes, n_bad);
  return 0;
}

// ================================================================================================================
// Accumulators
// ================================================================================================================
int vbgpu_acc_create(vbgpu_gmm_t model, vbgpu_acc_t *out) { return vbgpu_acc_create_with_transitions(model, 0, out); }

int vbgpu_acc_create_with_transitions(vbgpu_gmm_t model, int32_t num_tids, vbgpu_acc_t *out) {
  VB_CHECK(model && out && num_tids >= 0, "bad argument");
  *out = nullptr;
  DeviceGuard g(model->device);
  std::unique_ptr<vbgpu_acc_s, decltype(&vbgpu_acc_destroy)> h(new vbgpu_acc_s, vbgpu_acc_destroy);
  h->model = model;
  h->device = model->device;
  h->n_trans = num_tids > 0 ? num_tids + 1 : 0;  // indexed by the 1-based transition-id
  h->n_doubles = (int64_t)model->N * (2 * model->D + 1) + 2 + h->n_trans;
  VB_TRY(h->stream.create());
  VB_TRY(h->d_acc.reserve((size_t)h->n_doubles * 8));
  VB_CUDA(cudaMemset(h->d_acc.p, 0, (size_t)h->n_doubles * 8));
  *out = h.release();
  return 0;
}

int vbgpu_acc_destroy(vbgpu_acc_t h) {
  if (!h) return 0;
  DeviceGuard g(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  delete h;
  return 0;
}

int vbgpu_acc_zero(vbgpu_acc_t h) {
  VB_CHECK(h, "null handle");
  DeviceGuard g(h->device);
  VB_CUDA(cudaDeviceSynchronize());
  VB_CUDA(cudaMemset(h->d_acc.p, 0, (size_t)h->n_doubles * 8));
  return 0;
}

int vbgpu_acc_accumulate_dev(vbgpu_acc_t h, const float *d_feats, const float *d_feats2, int64_t T, int32_t stride,
                             const int32_t *d_pdf_ids, const float *d_weights, void *stream) {
  VB_CHECK(h && T >= 0, "bad argument");
  VB_CHECK(stride >= h->model->D, "stride %d < D %d", stride, h->model->D);
  if (T == 0) return 0;
  VB_CHECK(d_feats && d_pdf_ids, "null buffer");
  DeviceGuard g(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  VB_TRY(h->order.enter(s));  // the counting-sort work space of the bucketed accumulation
  VB_TRY(acc_launch(h, d_feats, d_feats2, T, stride, d_pdf_ids, d_weights, h->model->d_bad.as<unsigned long long>(), s));
  return h->order.leave(s);
}

int vbgpu_acc_accumulate(vbgpu_acc_t h, const float *feats, const float *feats2, int64_t T, int32_t stride,
                         const int32_t *pdf_ids, const float *weights, double *tot_like) {
  VB_CHECK(h && T >= 0, "bad argument");
  VB_CHECK(stride >= h->model->D, "stride %d < D %d", stride, h->model->D);
  if (tot_like) *tot_like = 0.0;
  if (T == 0) return 0;
  VB_CHECK(feats && pdf_ids, "null buffer");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  const size_t fb = (size_t)T * stride * 4;
  VB_TRY(h->d_feats.reserve(fb));
  VB_TRY(h->d_ids.reserve((size_t)T * 4));
  VB_TRY(h2d(h->d_feats.p, feats, fb, s));
  VB_TRY(h2d(h->d_ids.p, pdf_ids, (size_t)T * 4, s));
  const float *d_f2 = nullptr, *d_w = nullptr;
  if (feats2) {
    VB_TRY(h->d_feats2.reserve(fb));
    VB_TRY(h2d(h->d_feats2.p, feats2, fb, s));
    d_f2 = h->d_feats2.as<float>();
  }
  if (weights) {
    VB_TRY(h->d_w.reserve((size_t)T * 4));
    VB_TRY(h2d(h->d_w.p, weights, (size_t)T * 4, s));
    d_w = h->d_w.as<float>();
  }
  const size_t tail = (size_t)h->model->N * (2 * h->model->D + 1);
  double before = 0.0, after = 0.0;
  unsigned long long *bad = nullptr, n_bad = 0;
  VB_CUDA(cudaMemcpyAsync(&before, h->d_acc.as<double>() + tail, 8, cudaMemcpyDeviceToHost, s));
  VB_TRY(h->count.begin(s, &bad));
  VB_TRY(acc_launch(h, h->d_feats.as<float>(), d_f2, T, stride, h->d_ids.as<int32_t>(), d_w, bad, s));
  VB_CUDA(cudaMemcpyAsync(&after, h->d_acc.as<double>() + tail, 8, cudaMemcpyDeviceToHost, s));
  VB_TRY(h->count.end(s, &n_bad));
  if (tot_like) *tot_like = after - before;
  if (n_bad) return fail(VBGPU_ERR_NUMERIC, "%llu frames had an invalid pdf-id or a NaN/Inf likelihood", n_bad);
  return 0;
}

// The transition accumulators behind tot_frames in the statistics buffer.
static double *d_trans(vbgpu_acc_t h) { return h->d_acc.as<double>() + (size_t)h->model->N * (2 * h->model->D + 1) + 2; }

int vbgpu_acc_accumulate_transitions_dev(vbgpu_acc_t h, const int32_t *d_tids, int64_t T, void *stream) {
  VB_CHECK(h && T >= 0, "bad argument");
  VB_CHECK(h->n_trans > 0, "the accumulator was created without transition accumulators");
  if (T == 0) return 0;
  VB_CHECK(d_tids, "null buffer");
  DeviceGuard g(h->device);
  return acc_transitions_launch(d_trans(h), h->n_trans, d_tids, T, h->model->d_bad.as<unsigned long long>(),
                                static_cast<cudaStream_t>(stream));
}

int vbgpu_acc_accumulate_transitions(vbgpu_acc_t h, const int32_t *tids, int64_t T) {
  VB_CHECK(h && T >= 0, "bad argument");
  VB_CHECK(h->n_trans > 0, "the accumulator was created without transition accumulators");
  if (T == 0) return 0;
  VB_CHECK(tids, "null buffer");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  VB_TRY(h->d_ids.reserve((size_t)T * 4));
  unsigned long long *bad = nullptr, n_bad = 0;
  VB_TRY(h->count.begin(s, &bad));
  VB_TRY(h2d(h->d_ids.p, tids, (size_t)T * 4, s));
  VB_TRY(acc_transitions_launch(d_trans(h), h->n_trans, h->d_ids.as<int32_t>(), T, bad, s));
  VB_TRY(h->count.end(s, &n_bad));
  if (n_bad) return fail(VBGPU_ERR_INVALID, "%llu transition-ids outside [1, %d]", n_bad, h->n_trans - 1);
  return 0;
}

int vbgpu_acc_download_transitions(vbgpu_acc_t h, double *trans_accs) {
  VB_CHECK(h && trans_accs, "null argument");
  VB_CHECK(h->n_trans > 0, "the accumulator was created without transition accumulators");
  DeviceGuard g(h->device);
  VB_CUDA(cudaDeviceSynchronize());
  VB_CUDA(cudaMemcpy(trans_accs, d_trans(h), (size_t)h->n_trans * 8, cudaMemcpyDeviceToHost));
  return 0;
}

int vbgpu_acc_buffer(vbgpu_acc_t h, double **d_ptr, int64_t *n_doubles) {
  VB_CHECK(h && d_ptr && n_doubles, "null argument");
  *d_ptr = h->d_acc.as<double>();
  *n_doubles = h->n_doubles;
  return 0;
}

// In-place ncclAllReduce(ncclDouble, ncclSum) of n doubles on `device`.  libnccl is looked up at run time (already loaded
// by the caller, else dlopen), so the library has no link-time NCCL dependency.
static int nccl_allreduce_sum_f64(double *buf, int64_t n, int device, void *nccl_comm, void *stream) {
  typedef int (*allreduce_fn)(const void *, void *, size_t, int, int, void *, cudaStream_t);
  static allreduce_fn fn = nullptr;
  if (!fn) {
    fn = reinterpret_cast<allreduce_fn>(dlsym(RTLD_DEFAULT, "ncclAllReduce"));
    if (!fn) {
      void *lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
      if (lib) fn = reinterpret_cast<allreduce_fn>(dlsym(lib, "ncclAllReduce"));
    }
    if (!fn) return fail(VBGPU_ERR_INVALID, "ncclAllReduce not found: load libnccl.so.2 before calling");
  }
  DeviceGuard g(device);
  const int ncclDouble = 8, ncclSum = 0;
  int rc = fn(buf, buf, (size_t)n, ncclDouble, ncclSum, nccl_comm, static_cast<cudaStream_t>(stream));
  if (rc != 0) return fail(VBGPU_ERR_CUDA, "ncclAllReduce returned %d", rc);
  return 0;
}

int vbgpu_acc_allreduce(vbgpu_acc_t h, void *nccl_comm, void *stream) {
  VB_CHECK(h && nccl_comm, "null argument");
  return nccl_allreduce_sum_f64(h->d_acc.as<double>(), h->n_doubles, h->device, nccl_comm, stream);
}

int vbgpu_acc_add(vbgpu_acc_t h, double scale, vbgpu_acc_t other) {
  VB_CHECK(h && other, "null argument");
  VB_CHECK(h->n_doubles == other->n_doubles && h->device == other->device, "accumulators do not match");
  DeviceGuard g(h->device);
  VB_CUDA(cudaDeviceSynchronize());
  VB_TRY(acc_axpy(h->d_acc.as<double>(), other->d_acc.as<double>(), scale, h->n_doubles, h->stream));
  VB_CUDA(cudaStreamSynchronize(h->stream));
  return 0;
}

int vbgpu_acc_download(vbgpu_acc_t h, double *occ, double *mean_acc, double *var_acc, double *tot_like,
                       double *tot_frames) {
  VB_CHECK(h, "null handle");
  DeviceGuard g(h->device);
  VB_CUDA(cudaDeviceSynchronize());
  const size_t N = h->model->N, D = h->model->D;
  const double *a = h->d_acc.as<double>();
  if (occ) VB_CUDA(cudaMemcpy(occ, a, N * 8, cudaMemcpyDeviceToHost));
  if (mean_acc) VB_CUDA(cudaMemcpy(mean_acc, a + N, N * D * 8, cudaMemcpyDeviceToHost));
  if (var_acc) VB_CUDA(cudaMemcpy(var_acc, a + N + N * D, N * D * 8, cudaMemcpyDeviceToHost));
  double tail[2];
  VB_CUDA(cudaMemcpy(tail, a + N + 2 * N * D, 16, cudaMemcpyDeviceToHost));
  if (tot_like) *tot_like = tail[0];
  if (tot_frames) *tot_frames = tail[1];
  return 0;
}

// ================================================================================================================
// LDA class statistics
// ================================================================================================================
int vbgpu_lda_create(int32_t num_classes, int32_t dim, int device, vbgpu_lda_t *out) {
  VB_CHECK(out, "null argument");
  *out = nullptr;
  VB_CHECK(num_classes >= 1, "num_classes %d < 1", num_classes);
  VB_CHECK(dim >= 1 && dim <= 256, "dim %d outside 1 ... 256", dim);
  VB_TRY(check_device(device));
  DeviceGuard g(device);
  std::unique_ptr<vbgpu_lda_s, decltype(&vbgpu_lda_destroy)> h(new vbgpu_lda_s, vbgpu_lda_destroy);
  h->device = device;
  h->C = num_classes;
  h->D = dim;
  h->n_doubles = (int64_t)num_classes * (dim + 1) + (int64_t)dim * (dim + 1) / 2;
  VB_TRY(h->stream.create());
  VB_TRY(h->d_acc.reserve((size_t)h->n_doubles * 8));
  VB_TRY(h->d_bad.reserve(8));
  VB_CUDA(cudaMemset(h->d_acc.p, 0, (size_t)h->n_doubles * 8));
  VB_CUDA(cudaMemset(h->d_bad.p, 0, 8));
  *out = h.release();
  return 0;
}

int vbgpu_lda_destroy(vbgpu_lda_t h) {
  if (!h) return 0;
  DeviceGuard g(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  delete h;
  return 0;
}

int vbgpu_lda_zero(vbgpu_lda_t h) {
  VB_CHECK(h, "null handle");
  DeviceGuard g(h->device);
  VB_CUDA(cudaDeviceSynchronize());
  VB_CUDA(cudaMemset(h->d_acc.p, 0, (size_t)h->n_doubles * 8));
  return 0;
}

static int check_lda_args(vbgpu_lda_t h, const float *feats, int64_t T, int32_t stride, const int32_t *ids) {
  VB_CHECK(h && T >= 0, "bad argument");
  VB_CHECK(stride >= h->D, "stride %d < dim %d", stride, h->D);
  VB_CHECK(T == 0 || (feats && ids), "null buffer");
  return 0;
}

int vbgpu_lda_accumulate_dev(vbgpu_lda_t h, const float *d_feats, int64_t T, int32_t stride, const int32_t *d_class_ids,
                             const float *d_weights, void *stream) {
  VB_TRY(check_lda_args(h, d_feats, T, stride, d_class_ids));
  if (T == 0) return 0;
  DeviceGuard g(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  VB_TRY(h->order.enter(s));  // the counting-sort work space
  VB_TRY(lda_launch(h, d_feats, T, stride, d_class_ids, d_weights, h->d_bad.as<unsigned long long>(), s));
  return h->order.leave(s);
}

int vbgpu_lda_accumulate(vbgpu_lda_t h, const float *feats, int64_t T, int32_t stride, const int32_t *class_ids,
                         const float *weights) {
  VB_TRY(check_lda_args(h, feats, T, stride, class_ids));
  if (T == 0) return 0;
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  VB_TRY(h->order.enter(s));
  const size_t fb = (size_t)T * stride * 4;
  VB_TRY(h->d_feats.reserve(fb));
  VB_TRY(h->d_ids.reserve((size_t)T * 4));
  VB_TRY(h2d(h->d_feats.p, feats, fb, s));
  VB_TRY(h2d(h->d_ids.p, class_ids, (size_t)T * 4, s));
  const float *d_w = nullptr;
  if (weights) {
    VB_TRY(h->d_w.reserve((size_t)T * 4));
    VB_TRY(h2d(h->d_w.p, weights, (size_t)T * 4, s));
    d_w = h->d_w.as<float>();
  }
  unsigned long long *bad = nullptr, n_bad = 0;
  VB_TRY(h->count.begin(s, &bad));
  VB_TRY(lda_launch(h, h->d_feats.as<float>(), T, stride, h->d_ids.as<int32_t>(), d_w, bad, s));
  VB_TRY(h->count.end(s, &n_bad));
  VB_TRY(h->order.leave(s));
  if (n_bad) return fail(VBGPU_ERR_NUMERIC, "%llu frames had a class id outside [0, %d)", n_bad, h->C);
  return 0;
}

int vbgpu_lda_bad_count(vbgpu_lda_t h, int64_t *count) {
  VB_CHECK(h && count, "null argument");
  DeviceGuard g(h->device);
  VB_CUDA(cudaDeviceSynchronize());
  unsigned long long v = 0;
  VB_CUDA(cudaMemcpy(&v, h->d_bad.p, 8, cudaMemcpyDeviceToHost));
  VB_CUDA(cudaMemset(h->d_bad.p, 0, 8));
  *count = (int64_t)v;
  return 0;
}

int vbgpu_lda_download(vbgpu_lda_t h, double *zero, double *first, double *second) {
  VB_CHECK(h, "null handle");
  DeviceGuard g(h->device);
  VB_CUDA(cudaDeviceSynchronize());
  const size_t C = h->C, D = h->D;
  const double *a = h->d_acc.as<double>();
  if (zero) VB_CUDA(cudaMemcpy(zero, a, C * 8, cudaMemcpyDeviceToHost));
  if (first) VB_CUDA(cudaMemcpy(first, a + C, C * D * 8, cudaMemcpyDeviceToHost));
  if (second) VB_CUDA(cudaMemcpy(second, a + C + C * D, D * (D + 1) / 2 * 8, cudaMemcpyDeviceToHost));
  return 0;
}

int vbgpu_lda_buffer(vbgpu_lda_t h, double **d_ptr, int64_t *n_doubles) {
  VB_CHECK(h && d_ptr && n_doubles, "null argument");
  *d_ptr = h->d_acc.as<double>();
  *n_doubles = h->n_doubles;
  return 0;
}

int vbgpu_lda_allreduce(vbgpu_lda_t h, void *nccl_comm, void *stream) {
  VB_CHECK(h && nccl_comm, "null argument");
  return nccl_allreduce_sum_f64(h->d_acc.as<double>(), h->n_doubles, h->device, nccl_comm, stream);
}

// ================================================================================================================
// Tree statistics (kernels and the key layout in tree.cu)
// ================================================================================================================
int vbgpu_tree_create(const vbgpu_tree_opts *opts, const vbgpu_tid_tables *tables, int32_t dim, int32_t max_keys,
                      int device, vbgpu_tree_t *out) {
  VB_CHECK(out, "null argument");
  *out = nullptr;
  VB_TRY(tree_check(opts, tables, dim, max_keys));
  VB_TRY(check_device(device));
  DeviceGuard g(device);
  std::unique_ptr<vbgpu_tree_s, decltype(&vbgpu_tree_destroy)> h(new vbgpu_tree_s, vbgpu_tree_destroy);
  h->device = device;
  h->D = dim;
  h->max_keys = max_keys;
  VB_TRY(h->stream.create());
  VB_TRY(tree_init(h.get(), opts, tables));
  *out = h.release();
  return 0;
}

int vbgpu_tree_destroy(vbgpu_tree_t h) {
  if (!h) return 0;
  DeviceGuard g(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  delete h;
  return 0;
}

int vbgpu_tree_zero(vbgpu_tree_t h) {
  VB_CHECK(h, "null handle");
  DeviceGuard g(h->device);
  VB_CUDA(cudaDeviceSynchronize());
  return tree_zero(h, h->stream);
}

static int check_tree_args(vbgpu_tree_t h, const float *feats, int32_t stride, const int32_t *tids,
                           const int64_t *frame_offsets, int32_t n_utts) {
  VB_CHECK(h && n_utts >= 0, "bad argument");
  VB_CHECK(stride >= h->D, "stride %d < dim %d", stride, h->D);
  VB_CHECK(n_utts == 0 || frame_offsets, "null frame_offsets");
  if (n_utts == 0) return 0;
  VB_CHECK(frame_offsets[0] == 0, "frame_offsets[0] = %lld, not 0", (long long)frame_offsets[0]);
  for (int32_t u = 0; u < n_utts; u++)
    VB_CHECK(frame_offsets[u + 1] >= frame_offsets[u], "frame_offsets not monotone at utterance %d", u);
  VB_CHECK(frame_offsets[n_utts] == 0 || (feats && tids), "null buffer");
  return 0;
}

int vbgpu_tree_accumulate_dev(vbgpu_tree_t h, const float *d_feats, int32_t stride, const int32_t *d_tids,
                              const int64_t *frame_offsets, int32_t n_utts, void *stream) {
  VB_TRY(check_tree_args(h, d_feats, stride, d_tids, frame_offsets, n_utts));
  if (n_utts == 0) return 0;
  DeviceGuard g(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  VB_TRY(h->order.enter(s));
  VB_TRY(h->layout.update(nullptr, frame_offsets, n_utts, nullptr, nullptr, s));
  VB_TRY(tree_launch(h, d_feats, stride, d_tids, h->layout.d_frame_offsets.as<int64_t>(), n_utts, h->layout.total_frames,
                     s));
  return h->order.leave(s);
}

int vbgpu_tree_accumulate(vbgpu_tree_t h, const float *feats, int32_t stride, const int32_t *tids,
                          const int64_t *frame_offsets, int32_t n_utts) {
  VB_TRY(check_tree_args(h, feats, stride, tids, frame_offsets, n_utts));
  if (n_utts == 0) return 0;
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  VB_TRY(h->order.enter(s));
  const int64_t T = frame_offsets[n_utts];
  VB_TRY(h->d_feats.reserve((size_t)std::max<int64_t>(T, 1) * stride * 4));
  VB_TRY(h->d_tids.reserve((size_t)std::max<int64_t>(T, 1) * 4));
  VB_TRY(h2d(h->d_feats.p, feats, (size_t)T * stride * 4, s));
  VB_TRY(h2d(h->d_tids.p, tids, (size_t)T * 4, s));
  int64_t before = 0, after = 0;
  VB_CUDA(cudaStreamSynchronize(s));
  VB_TRY(tree_counters(h, nullptr, &before, nullptr, false));
  VB_TRY(h->layout.update(nullptr, frame_offsets, n_utts, nullptr, nullptr, s));
  VB_TRY(tree_launch(h, h->d_feats.as<float>(), stride, h->d_tids.as<int32_t>(), h->layout.d_frame_offsets.as<int64_t>(),
                     n_utts, T, s));
  VB_CUDA(cudaStreamSynchronize(s));
  VB_TRY(tree_counters(h, nullptr, &after, nullptr, false));
  VB_TRY(h->order.leave(s));
  if (after != before)
    return fail(VBGPU_ERR_NUMERIC, "%lld frames found no room in the key table (max_keys %d)", (long long)(after - before),
                h->max_keys);
  return 0;
}

int vbgpu_tree_bad_count(vbgpu_tree_t h, int64_t *bad_utterances, int64_t *dropped_frames) {
  VB_CHECK(h, "null handle");
  DeviceGuard g(h->device);
  VB_CUDA(cudaDeviceSynchronize());
  return tree_counters(h, bad_utterances, dropped_frames, nullptr, true);
}

int vbgpu_tree_num_keys(vbgpu_tree_t h, int32_t *num_keys) {
  VB_CHECK(h && num_keys, "null argument");
  DeviceGuard g(h->device);
  VB_CUDA(cudaDeviceSynchronize());
  int64_t k = 0;
  VB_TRY(tree_counters(h, nullptr, nullptr, &k, false));
  *num_keys = (int32_t)k;
  return 0;
}

int vbgpu_tree_download(vbgpu_tree_t h, int32_t *pdf_class, int32_t *phones, double *count, double *sum_x,
                        double *sum_x2) {
  VB_CHECK(h, "null handle");
  DeviceGuard g(h->device);
  VB_CUDA(cudaDeviceSynchronize());
  return tree_download(h, pdf_class, phones, count, sum_x, sum_x2);
}

int vbgpu_tree_add(vbgpu_tree_t h, int32_t n, const int32_t *pdf_class, const int32_t *phones, const double *count,
                   const double *sum_x, const double *sum_x2) {
  VB_CHECK(h && n >= 0, "bad argument");
  VB_CHECK(n == 0 || (pdf_class && phones && count && sum_x && sum_x2), "null buffer");
  DeviceGuard g(h->device);
  VB_CUDA(cudaDeviceSynchronize());
  int64_t dropped = 0;
  VB_TRY(tree_add(h, n, pdf_class, phones, count, sum_x, sum_x2, &dropped));
  if (dropped)
    return fail(VBGPU_ERR_NUMERIC, "%lld entries found no room in the key table (max_keys %d)", (long long)dropped,
                h->max_keys);
  return 0;
}

// ================================================================================================================
// Fused pipelines
// ================================================================================================================
int vbgpu_pipeline_create(vbgpu_mfcc_t mfcc, vbgpu_feat_t feat, vbgpu_gmm_t gmm, vbgpu_pipeline_t *out) {
  VB_CHECK(mfcc && feat && gmm && out, "null argument");
  *out = nullptr;
  VB_CHECK(mfcc->device == feat->device && feat->device == gmm->device, "handles live on different devices");
  VB_CHECK(feat->in_dim == feat_dim_of(mfcc), "feature pipeline expects dim %d, the front end gives %d", feat->in_dim,
           feat_dim_of(mfcc));
  VB_CHECK(feat->out_dim == gmm->D, "feature pipeline gives dim %d, model expects %d", feat->out_dim, gmm->D);
  DeviceGuard g(gmm->device);
  std::unique_ptr<vbgpu_pipeline_s, decltype(&vbgpu_pipeline_destroy)> h(new vbgpu_pipeline_s, vbgpu_pipeline_destroy);
  h->mfcc = mfcc;
  h->feat = feat;
  h->gmm = gmm;
  h->device = gmm->device;
  VB_TRY(h->stream.create());
  VB_TRY(h->copy_stream.create());
  for (int i = 0; i < 2; i++) {
    VB_TRY(h->ev_ll[i].create());
    VB_TRY(h->ev_copied[i].create());
  }
  *out = h.release();
  return 0;
}

int vbgpu_pipeline_destroy(vbgpu_pipeline_t h) {
  if (!h) return 0;
  DeviceGuard g(h->device);
  cudaDeviceSynchronize();
  delete h;
  return 0;
}

// PCM (device) -> processed features (device), all on stream s.  d_stats_in: precomputed per-speaker stats or null.
static int pipeline_front(vbgpu_pipeline_t h, const int16_t *d_pcm, const int64_t *sample_offsets, int32_t n_utts,
                          const int32_t *utt2spk, int32_t n_spk, const double *d_stats_in, bool check_stats,
                          const float *d_fmllr, int32_t fmllr_cols, float *d_feats, int32_t feats_stride,
                          cudaStream_t s) {
  vbgpu_mfcc_t m = h->mfcc;
  vbgpu_feat_t f = h->feat;
  VB_TRY(h->order.enter(s));  // batch layouts, MFCC / statistics scratch of the three handles: see StreamOrder
  VB_TRY(m->order.enter(s));
  VB_TRY(f->order.enter(s));
  VB_TRY(check_spk(utt2spk, n_utts, n_spk));
  VB_TRY(check_fmllr(f, d_fmllr, fmllr_cols));
  VB_TRY(mfcc_prepare(m, sample_offsets, n_utts, nullptr, s));
  const int64_t T = m->layout.total_frames;
  VB_TRY(f->layout.update(nullptr, m->layout.h_frame_offsets.data(), n_utts, utt2spk, nullptr, s));
  if (T == 0) return 0;
  const int C = feat_dim_of(m), mst = (C + 3) / 4 * 4;
  VB_TRY(h->d_mfcc.reserve((size_t)T * mst * 4));
  VB_TRY(mfcc_launch(m, d_pcm, false, h->d_mfcc.as<float>(), mst, s));
  if (f->opts.norm_means || f->opts.norm_vars) {
    const double *d_stats = d_stats_in;
    if (!d_stats) {
      const size_t nst = (size_t)n_spk * 2 * (C + 1);
      VB_TRY(f->d_stats.reserve(nst * 8));
      VB_CUDA(cudaMemsetAsync(f->d_stats.p, 0, nst * 8, s));
      VB_TRY(feat_launch_stats(f, h->d_mfcc.as<float>(), mst, f->d_stats.as<double>(), n_spk, s));
      d_stats = f->d_stats.as<double>();
    }
    VB_TRY(feat_norm_from_stats(f, d_stats, n_spk, check_stats, s));
  }
  VB_TRY(feat_launch(f, h->d_mfcc.as<float>(), mst, d_fmllr, fmllr_cols, d_feats, feats_stride, s));
  VB_TRY(m->order.leave(s));
  VB_TRY(f->order.leave(s));
  return h->order.leave(s);
}

static int pipeline_score_dev(vbgpu_pipeline_t h, const int16_t *d_pcm, const int64_t *sample_offsets, int32_t n_utts,
                              const int32_t *utt2spk, int32_t n_spk, const float *d_fmllr, int32_t fmllr_cols,
                              float *d_loglikes, int32_t ll_stride, float *d_feats, int32_t feats_stride, int native,
                              void *stream) {
  VB_CHECK(h && sample_offsets && n_utts >= 0, "bad argument");
  const int need = native ? native_cols(h->gmm) : h->gmm->P;
  VB_CHECK(ll_stride >= need, "ll_stride %d < %d columns", ll_stride, need);
  if (n_utts == 0) return 0;
  VB_CHECK(sample_offsets[0] == 0, "sample_offsets[0] must be 0");
  DeviceGuard g(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int D = h->gmm->D;
  float *feats = d_feats;
  int32_t fst = feats_stride;
  if (!feats) {
    fst = (D + 3) / 4 * 4;
    int64_t T = 0;
    for (int32_t u = 0; u < n_utts; u++) T += num_frames_of(h->mfcc, sample_offsets[u + 1] - sample_offsets[u]);
    VB_TRY(h->d_feats.reserve((size_t)std::max<int64_t>(T, 1) * fst * 4));
    feats = h->d_feats.as<float>();
  } else {
    VB_CHECK(fst >= D, "feats_stride %d < D %d", fst, D);
  }
  VB_TRY(pipeline_front(h, d_pcm, sample_offsets, n_utts, utt2spk, n_spk, nullptr, false, d_fmllr, fmllr_cols, feats,
                        fst, s));
  const int64_t T = h->mfcc->layout.total_frames;
  if (T == 0) return 0;
  VB_CHECK(d_pcm && d_loglikes, "null buffer");
  return score_dispatch(h->gmm, feats, T, fst, d_loglikes, ll_stride, native != 0, h->gmm->d_bad.as<unsigned long long>(),
                        s);
}

int vbgpu_pipeline_score_dev(vbgpu_pipeline_t h, const int16_t *d_pcm, const int64_t *sample_offsets, int32_t n_utts,
                             const int32_t *utt2spk, int32_t n_spk, const float *d_fmllr, int32_t fmllr_cols,
                             float *d_loglikes, int32_t ll_stride, float *d_feats, int32_t feats_stride, void *stream) {
  return pipeline_score_dev(h, d_pcm, sample_offsets, n_utts, utt2spk, n_spk, d_fmllr, fmllr_cols, d_loglikes, ll_stride,
                            d_feats, feats_stride, 0, stream);
}

int vbgpu_pipeline_score_cols_dev(vbgpu_pipeline_t h, const int16_t *d_pcm, const int64_t *sample_offsets, int32_t n_utts,
                                  const int32_t *utt2spk, int32_t n_spk, const float *d_fmllr, int32_t fmllr_cols,
                                  float *d_loglikes, int32_t ll_stride, float *d_feats, int32_t feats_stride,
                                  void *stream) {
  return pipeline_score_dev(h, d_pcm, sample_offsets, n_utts, utt2spk, n_spk, d_fmllr, fmllr_cols, d_loglikes, ll_stride,
                            d_feats, feats_stride, 1, stream);
}

int vbgpu_pipeline_accumulate_dev(vbgpu_pipeline_t h, vbgpu_acc_t acc, const int16_t *d_pcm,
                                  const int64_t *sample_offsets, int32_t n_utts, const int32_t *utt2spk, int32_t n_spk,
                                  const float *d_fmllr, int32_t fmllr_cols, const int32_t *d_pdf_ids, void *stream) {
  VB_CHECK(h && acc && sample_offsets && n_utts >= 0, "bad argument");
  VB_CHECK(acc->model == h->gmm, "accumulator belongs to a different model");
  VB_TRY(acc->order.enter(static_cast<cudaStream_t>(stream)));
  if (n_utts == 0) return 0;
  VB_CHECK(sample_offsets[0] == 0, "sample_offsets[0] must be 0");
  DeviceGuard g(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int D = h->gmm->D, fst = (D + 3) / 4 * 4;
  int64_t T = 0;
  for (int32_t u = 0; u < n_utts; u++) T += num_frames_of(h->mfcc, sample_offsets[u + 1] - sample_offsets[u]);
  VB_TRY(h->d_feats.reserve((size_t)std::max<int64_t>(T, 1) * fst * 4));
  VB_TRY(pipeline_front(h, d_pcm, sample_offsets, n_utts, utt2spk, n_spk, nullptr, false, d_fmllr, fmllr_cols,
                        h->d_feats.as<float>(), fst, s));
  if (T == 0) return 0;
  VB_CHECK(d_pcm && d_pdf_ids, "null buffer");
  VB_TRY(acc_launch(acc, h->d_feats.as<float>(), nullptr, T, fst, d_pdf_ids, nullptr,
                    acc->model->d_bad.as<unsigned long long>(), s));
  VB_TRY(h->order.leave(s));  // (h->d_feats is read by the accumulation kernels)
  return acc->order.leave(s);
}

// Host PCM -> processed features in h->d_feats (stride (D+3)/4*4), everything enqueued on the pipeline's stream.
// Pinned caller buffers are DMA sources directly; pageable ones go through pinned staging.
static int pipeline_host_front(vbgpu_pipeline_t h, const int16_t *pcm, const int64_t *sample_offsets, int32_t n_utts,
                               const int32_t *utt2spk, int32_t n_spk, const double *cmvn_stats, const float *fmllr,
                               int32_t fmllr_cols, int64_t *T_out) {
  const int D = h->gmm->D;
  cudaStream_t s = h->stream;
  const int64_t ns = sample_offsets[n_utts];
  int64_t T = 0;
  for (int32_t u = 0; u < n_utts; u++) T += num_frames_of(h->mfcc, sample_offsets[u + 1] - sample_offsets[u]);
  *T_out = T;
  const int fst = (D + 3) / 4 * 4;
  VB_TRY(h->d_pcm.reserve((size_t)std::max<int64_t>(ns, 1) * 2));
  if (is_pinned_or_device(pcm)) {
    VB_TRY(h2d(h->d_pcm.p, pcm, (size_t)ns * 2, s));
  } else {  // pageable: stage through pinned memory in 32 MiB pieces so the DMA engine never waits on a page fault
    const size_t piece = 32u << 20;
    VB_TRY(h->pin_pcm.reserve(2 * piece));
    size_t done = 0;
    int k = 0;
    cudaEvent_t ev[2] = {h->ev_copied[0], h->ev_copied[1]};
    bool used[2] = {false, false};
    while (done < (size_t)ns * 2) {
      const size_t n = std::min(piece, (size_t)ns * 2 - done);
      if (used[k]) VB_CUDA(cudaEventSynchronize(ev[k]));
      std::memcpy(h->pin_pcm.as<char>() + k * piece, reinterpret_cast<const char *>(pcm) + done, n);
      VB_CUDA(cudaMemcpyAsync(h->d_pcm.as<char>() + done, h->pin_pcm.as<char>() + k * piece, n, cudaMemcpyHostToDevice, s));
      VB_CUDA(cudaEventRecord(ev[k], s));
      used[k] = true;
      done += n;
      k ^= 1;
    }
  }
  const double *d_stats = nullptr;
  if (cmvn_stats && (h->feat->opts.norm_means || h->feat->opts.norm_vars)) {
    const size_t nst = (size_t)n_spk * 2 * (h->feat->in_dim + 1);
    VB_TRY(h->d_stats.reserve(nst * 8));
    VB_TRY(h2d(h->d_stats.p, cmvn_stats, nst * 8, s));
    d_stats = h->d_stats.as<double>();
  }
  const float *d_fm = nullptr;
  if (fmllr) {
    VB_CHECK(fmllr_cols == D || fmllr_cols == D + 1, "fMLLR matrix has %d columns, feature dim is %d", fmllr_cols, D);
    const size_t nb = (size_t)n_spk * D * fmllr_cols * 4;
    VB_TRY(h->d_fmllr.reserve(nb));
    VB_TRY(h2d(h->d_fmllr.p, fmllr, nb, s));
    d_fm = h->d_fmllr.as<float>();
  }
  VB_TRY(h->d_feats.reserve((size_t)std::max<int64_t>(T, 1) * fst * 4));
  return pipeline_front(h, h->d_pcm.as<int16_t>(), sample_offsets, n_utts, utt2spk, n_spk, d_stats, true, d_fm, fmllr_cols,
                        h->d_feats.as<float>(), fst, s);
}

// Host form: H2D of the PCM, front end, then scoring in slabs of frames whose D2H copies overlap the next slab's
// kernel (two device slabs, two events per slab).
int vbgpu_pipeline_score_i16(vbgpu_pipeline_t h, const int16_t *pcm, const int64_t *sample_offsets, int32_t n_utts,
                             const int32_t *utt2spk, int32_t n_spk, const double *cmvn_stats, const float *fmllr,
                             int32_t fmllr_cols, float *loglikes, int32_t ll_stride, float *feats_out,
                             int32_t feats_stride) {
  VB_CHECK(h && sample_offsets && n_utts >= 0, "bad argument");
  const int P = h->gmm->P, D = h->gmm->D;
  VB_CHECK(ll_stride >= P, "ll_stride %d < P %d", ll_stride, P);
  VB_CHECK(!feats_out || feats_stride >= D, "feats_stride %d < D %d", feats_stride, D);
  if (n_utts == 0) return 0;
  VB_CHECK(sample_offsets[0] == 0, "sample_offsets[0] must be 0");
  VB_CHECK(pcm, "null pcm");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream, cs = h->copy_stream;
  const int fst = (D + 3) / 4 * 4;
  int64_t T = 0;
  VB_TRY(pipeline_host_front(h, pcm, sample_offsets, n_utts, utt2spk, n_spk, cmvn_stats, fmllr, fmllr_cols, &T));
  if (T == 0) return 0;
  VB_CHECK(loglikes, "null loglikes");
  if (feats_out) {
    VB_CUDA(cudaMemcpy2DAsync(feats_out, (size_t)feats_stride * 4, h->d_feats.p, (size_t)fst * 4, (size_t)D * 4, T,
                              cudaMemcpyDeviceToHost, s));
  }

  // ---- scoring slabs, D2H overlapped ----
  int64_t slab = (int64_t)(256ull << 20) / ((int64_t)ll_stride * 4);
  slab = std::max<int64_t>(256, slab / 256 * 256);
  slab = std::min(slab, T);
  const size_t slab_bytes = (size_t)slab * ll_stride * 4;
  const bool direct = is_pinned_or_device(loglikes);
  for (int i = 0; i < 2; i++) {
    VB_TRY(h->d_ll[i].reserve(slab_bytes));
    if (!direct) VB_TRY(h->pin_ll[i].reserve(slab_bytes));
  }
  unsigned long long *bad = nullptr, n_bad = 0;
  VB_TRY(h->count.begin(s, &bad));
  bool inflight[2] = {false, false};
  int64_t pend_t0[2] = {0, 0}, pend_n[2] = {0, 0};
  int k = 0;
  for (int64_t t0 = 0; t0 < T; t0 += slab, k ^= 1) {
    const int64_t n = std::min(slab, T - t0);
    if (inflight[k]) {  // the slab buffer is being copied out: wait, then (pageable) drain the staging buffer
      VB_CUDA(cudaEventSynchronize(h->ev_copied[k]));
      if (!direct)
        std::memcpy(loglikes + pend_t0[k] * ll_stride, h->pin_ll[k].p, (size_t)pend_n[k] * ll_stride * 4);
      inflight[k] = false;
    }
    VB_TRY(score_dispatch(h->gmm, h->d_feats.as<float>() + t0 * fst, n, fst, h->d_ll[k].as<float>(), ll_stride, false, bad,
                          s));
    VB_CUDA(cudaEventRecord(h->ev_ll[k], s));
    VB_CUDA(cudaStreamWaitEvent(cs, h->ev_ll[k], 0));
    void *dst = direct ? static_cast<void *>(loglikes + t0 * ll_stride) : h->pin_ll[k].p;
    VB_CUDA(cudaMemcpyAsync(dst, h->d_ll[k].p, (size_t)n * ll_stride * 4, cudaMemcpyDeviceToHost, cs));
    VB_CUDA(cudaEventRecord(h->ev_copied[k], cs));
    inflight[k] = true;
    pend_t0[k] = t0;
    pend_n[k] = n;
  }
  for (int i = 0; i < 2; i++) {
    const int j = k ^ i;  // older slab first
    if (inflight[j]) {
      VB_CUDA(cudaEventSynchronize(h->ev_copied[j]));
      if (!direct) std::memcpy(loglikes + pend_t0[j] * ll_stride, h->pin_ll[j].p, (size_t)pend_n[j] * ll_stride * 4);
    }
  }
  VB_TRY(h->count.end(s, &n_bad));
  if (n_bad) return fail(VBGPU_ERR_NUMERIC, kBadLoglikes, n_bad);
  return 0;
}

// PCM (host) -> the log-likelihoods forced alignment reads: utterance u's own pdf subset (gmm-align-compiled.cpp:119-128).
int vbgpu_pipeline_score_subset_i16(vbgpu_pipeline_t h, const int16_t *pcm, const int64_t *sample_offsets, int32_t n_utts,
                                    const int32_t *utt2spk, int32_t n_spk, const double *cmvn_stats, const float *fmllr,
                                    int32_t fmllr_cols, const int64_t *subset_offsets, const int32_t *subset_pdfs, float *out,
                                    int64_t *out_offsets) {
  VB_CHECK(h && sample_offsets && n_utts >= 1 && pcm, "bad argument");
  VB_CHECK(sample_offsets[0] == 0, "sample_offsets[0] must be 0");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  const int D = h->gmm->D, fst = (D + 3) / 4 * 4;
  int64_t T = 0;
  VB_TRY(pipeline_host_front(h, pcm, sample_offsets, n_utts, utt2spk, n_spk, cmvn_stats, fmllr, fmllr_cols, &T));
  SparseReq rq;
  int64_t total = 0;
  VB_TRY(sparse_prepare_subset(h->gmm, T, h->mfcc->layout.h_frame_offsets.data(), n_utts, subset_offsets, subset_pdfs,
                               out_offsets, &total, &rq, s));
  if (total == 0) return 0;
  VB_CHECK(out, "null output");
  VB_TRY(h->gmm->d_sp_out.reserve((size_t)total * 4));
  unsigned long long *bad = nullptr, n_bad = 0;
  VB_TRY(h->count.begin(s, &bad));
  rq.d_out = h->gmm->d_sp_out.as<float>();
  rq.h_out = out;  // results leave slab by slab, behind the scoring of the next slab
  VB_TRY(score_sparse_dev(h->gmm, h->d_feats.as<float>(), T, fst, rq, bad, s));
  VB_TRY(h->count.end(s, &n_bad));
  if (n_bad) return fail(VBGPU_ERR_NUMERIC, kBadLoglikes, n_bad);
  return 0;
}

// PCM (host) -> one log-likelihood per lattice arc: frames[] index the packed batch (lattice-functions.cc:1214-1360).
int vbgpu_pipeline_score_gather_i16(vbgpu_pipeline_t h, const int16_t *pcm, const int64_t *sample_offsets, int32_t n_utts,
                                    const int32_t *utt2spk, int32_t n_spk, const double *cmvn_stats, const float *fmllr,
                                    int32_t fmllr_cols, const int32_t *frames, const int32_t *pdfs, int64_t n, float *out) {
  VB_CHECK(h && sample_offsets && n_utts >= 1 && pcm, "bad argument");
  VB_CHECK(sample_offsets[0] == 0, "sample_offsets[0] must be 0");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  const int D = h->gmm->D, fst = (D + 3) / 4 * 4;
  int64_t T = 0;
  VB_TRY(pipeline_host_front(h, pcm, sample_offsets, n_utts, utt2spk, n_spk, cmvn_stats, fmllr, fmllr_cols, &T));
  SparseReq rq;
  VB_TRY(sparse_prepare_gather(h->gmm, T, frames, pdfs, n, &rq, s));
  if (n == 0) return 0;
  VB_CHECK(out, "null output");
  VB_TRY(h->gmm->d_sp_out.reserve((size_t)n * 4));
  unsigned long long *bad = nullptr, n_bad = 0;
  VB_TRY(h->count.begin(s, &bad));
  rq.d_out = h->gmm->d_sp_out.as<float>();
  VB_TRY(score_sparse_dev(h->gmm, h->d_feats.as<float>(), T, fst, rq, bad, s));
  VB_TRY(d2h(out, h->gmm->d_sp_out.p, (size_t)n * 4, s));
  VB_TRY(h->count.end(s, &n_bad));
  if (n_bad) return fail(VBGPU_ERR_NUMERIC, kBadLoglikes, n_bad);
  return 0;
}

}  // extern "C"
