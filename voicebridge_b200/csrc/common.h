// common.h — internal helpers shared by the libvbgpu translation units (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/vbgpu.h"

namespace vb {

// ---- error reporting: thread-local message, int codes across the ABI -----------------------------------
std::string &last_error();
int fail(int code, const char *fmt, ...);

#define VB_CUDA(expr)                                                                              \
  do {                                                                                             \
    cudaError_t e_ = (expr);                                                                       \
    if (e_ != cudaSuccess) return vb::fail(VBGPU_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e_)); \
  } while (0)

#define VB_CHECK(cond, ...)                                   \
  do {                                                        \
    if (!(cond)) return vb::fail(VBGPU_ERR_INVALID, __VA_ARGS__); \
  } while (0)

#define VB_TRY(expr)         \
  do {                       \
    int rc_ = (expr);        \
    if (rc_ < 0) return rc_; \
  } while (0)

// Fails with VBGPU_ERR_CUDA ("no CPU fallback") without a CUDA device, VBGPU_ERR_INVALID for a device out of range.
int check_device(int device);

// ---- owning handles of device memory, pinned memory, streams and events -----------------------------------------
// Bytes of device and pinned memory the library holds right now (vbgpu_debug_live_bytes): every cudaMalloc and
// cudaMallocHost goes through DevBuf / PinBuf.
inline std::atomic<int64_t> live_device_bytes{0}, live_pinned_bytes{0};

// Grow-only buffers, freed by their destructor.  A DevBuf is freed on the device that is current when its owner is
// destroyed, so a function declares its DeviceGuard before any local DevBuf, and a handle is deleted while a
// DeviceGuard for its device is alive.
struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  ~DevBuf() { release(); }
  int reserve(size_t bytes) {
    if (bytes <= cap) return 0;
    release();
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      p = nullptr;
      cudaGetLastError();  // reported here: the next launch check must not see this error again
      return fail(VBGPU_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
    }
    cap = want;
    live_device_bytes += (int64_t)want;
    return 0;
  }
  // reserve(bytes), then a synchronous copy of bytes from the host
  int upload(const void *src, size_t bytes) {
    int rc = reserve(bytes);
    if (rc < 0 || bytes == 0) return rc;
    cudaError_t e = cudaMemcpy(p, src, bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return fail(VBGPU_ERR_CUDA, "upload of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
    return 0;
  }
  template <typename T>
  T *as() const { return static_cast<T *>(p); }

 private:
  void release() {
    if (p) {
      cudaFree(p);
      live_device_bytes -= (int64_t)cap;
    }
    p = nullptr;
    cap = 0;
  }
};

struct PinBuf {
  void *p = nullptr;
  size_t cap = 0;
  PinBuf() = default;
  PinBuf(const PinBuf &) = delete;
  PinBuf &operator=(const PinBuf &) = delete;
  ~PinBuf() { release(); }
  int reserve(size_t bytes) {
    if (bytes <= cap) return 0;
    release();
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMallocHost(&p, want);
    if (e != cudaSuccess) {
      p = nullptr;
      cudaGetLastError();
      return fail(VBGPU_ERR_NOMEM, "cudaMallocHost(%zu) failed: %s", want, cudaGetErrorString(e));
    }
    cap = want;
    live_pinned_bytes += (int64_t)want;
    return 0;
  }
  template <typename T>
  T *as() const { return static_cast<T *>(p); }

 private:
  void release() {
    if (p) {
      cudaFreeHost(p);
      live_pinned_bytes -= (int64_t)cap;
    }
    p = nullptr;
    cap = 0;
  }
};

// A non-blocking stream, destroyed with its owner.  Converts to the raw handle (null until create()).
struct Stream {
  cudaStream_t s = nullptr;
  Stream() = default;
  Stream(const Stream &) = delete;
  Stream &operator=(const Stream &) = delete;
  ~Stream() {
    if (s) cudaStreamDestroy(s);
  }
  int create() {
    cudaError_t e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
      s = nullptr;
      return fail(VBGPU_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
    }
    return 0;
  }
  operator cudaStream_t() const { return s; }
};

// An event without timing, destroyed with its owner.  Converts to the raw handle (null until create()).
struct Event {
  cudaEvent_t ev = nullptr;
  Event() = default;
  Event(const Event &) = delete;
  Event &operator=(const Event &) = delete;
  ~Event() {
    if (ev) cudaEventDestroy(ev);
  }
  int create() {
    cudaError_t e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (e != cudaSuccess) {
      ev = nullptr;
      return fail(VBGPU_ERR_CUDA, "cudaEventCreate failed: %s", cudaGetErrorString(e));
    }
    return 0;
  }
  operator cudaEvent_t() const { return ev; }
};

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

int num_sms(int device);

// A handle's scratch buffers (batch layout, staging, statistics, work space) are re-used by every call.  Calls on ONE stream
// are ordered by the stream; a call on a different stream than the previous one must first wait for that one to finish with
// the scratch.  enter() makes the new stream wait on the event leave() recorded at the end of the previous call.
struct StreamOrder {
  cudaStream_t last = nullptr;
  Event ev;
  bool used = false;
  int enter(cudaStream_t s) {
    if (used && last != s) {
      cudaError_t e = cudaStreamWaitEvent(s, ev, 0);
      if (e != cudaSuccess) return fail(VBGPU_ERR_CUDA, "cudaStreamWaitEvent failed: %s", cudaGetErrorString(e));
    }
    return 0;
  }
  int leave(cudaStream_t s) {
    if (!ev) VB_TRY(ev.create());
    cudaError_t e = cudaEventRecord(ev, s);
    if (e != cudaSuccess) return fail(VBGPU_ERR_CUDA, "cudaEventRecord failed: %s", cudaGetErrorString(e));
    last = s;
    used = true;
    return 0;
  }
};

// ---- batch layout: the utterance structure of one packed batch, mirrored on the device ------------------------
// Cached by content: bench / training loops re-use the same layout every step and pay nothing.
struct BatchLayout {
  int32_t n_utts = 0;
  int64_t total_frames = 0, total_samples = 0;
  std::vector<int64_t> h_sample_offsets, h_frame_offsets;
  std::vector<int32_t> h_utt2spk, h_utt_aux;
  DevBuf d_sample_offsets, d_frame_offsets, d_frame2utt, d_utt2spk, d_utt_aux;
  PinBuf stage;
  // Upload (if changed) sample offsets + frame offsets and rebuild frame2utt.  utt2spk / utt_aux may be null.
  int update(const int64_t *sample_offsets, const int64_t *frame_offsets, int32_t n, const int32_t *utt2spk,
             const int32_t *utt_aux, cudaStream_t s);
};

void launch_fill_frame2utt(const int64_t *d_frame_offsets, int32_t n_utts, int64_t total_frames, int32_t *d_frame2utt,
                           cudaStream_t s);

}  // namespace vb

// ---- handle definitions -----------------------------------------------------------------------------------------
struct MelTable {  // one per distinct VTLN warp factor
  float warp;
};

struct vbgpu_mfcc_s {
  vb::StreamOrder order;  // cross-stream ordering of the handle's scratch (see StreamOrder)
  vbgpu_mfcc_opts opts;
  int device = 0;
  vb::Stream stream;
  int32_t L = 0, shift = 0, npad = 0, mel_pitch = 0;
  int32_t fbank = 0, use_log_fbank = 1, use_power = 1;  // fbank != 0: the handle is a FbankComputer (vbgpu_fbank_create)
  int32_t plp = 0, lpc_order = 12;                      // plp != 0: the handle is a PlpComputer (vbgpu_plp_create)
  float compress_factor = 0.33333f, cepstral_scale = 1.0f;
  vb::DevBuf d_idft, d_eq_loud;
  float log_energy_floor = 0.f;
  std::vector<float> warps;  // distinct VTLN factors with a table on the device (warps[0] == 1.0)
  vb::DevBuf d_window, d_tw, d_mel_off, d_mel_len, d_mel_w, d_dct, d_lifter;
  vb::DevBuf d_pcm, d_out;
  vb::PinBuf pin_in, pin_out;
  vb::BatchLayout layout;
  uint32_t dither_seed = 0x9E3779B9u;
};

struct vbgpu_feat_s {
  vb::StreamOrder order;  // cross-stream ordering of the handle's scratch (see StreamOrder)
  vbgpu_feat_opts opts;
  int device = 0;
  vb::Stream stream;
  int32_t in_dim = 0, mid_dim = 0, out_dim = 0, halo = 0;
  int32_t t_rows = 0, t_cols = 0;  // global transform (lda mode)
  std::vector<float> h_delta_scales;
  std::vector<int32_t> h_delta_lens;
  vb::DevBuf d_transform, d_delta_scales, d_norm, d_stats, d_fmllr, d_in, d_out;
  vb::BatchLayout layout;
};

struct vbgpu_gmm_s {
  vb::StreamOrder order;  // cross-stream ordering of the handle's scratch (see StreamOrder)
  int device = 0;
  vb::Stream stream;
  int32_t P = 0, N = 0, D = 0, DP = 0;  // DP: padded row length of the SIMT layout (multiple of 4)
  int32_t kernel = 0;
  int32_t max_pdf_size = 0;
  std::vector<int32_t> h_pdf_offsets;
  vb::DevBuf d_pdf_offsets, d_gconsts, d_rows;  // d_rows: [N][2*DP] = means_invvars | -0.5*inv_vars
  vb::DevBuf d_bad;                             // int64 counter of NaN/Inf outputs
  vb::DevBuf d_feats, d_ll;
  vb::DevBuf d_sp_slab, d_sp_i64, d_sp_i32, d_sp_f2u, d_sp_out;  // sparse consumers (score_sparse.cu): slab + descriptors
  vb::Stream copy_stream;  // host-facing subset calls: results of slab k leave while slab k+1 is scored
  vb::Event sp_done[2];
  void *tc = nullptr;  // tensor-core scoring state (score_tc.cu)
  std::string tc_note;  // why the model is NOT on the tensor-core plan ("" when it is)
};

struct vbgpu_acc_s {
  vb::StreamOrder order;  // cross-stream ordering of the handle's scratch (see StreamOrder)
  vbgpu_gmm_t model = nullptr;
  int device = 0;
  vb::Stream stream;
  int64_t n_doubles = 0;
  int32_t n_trans = 0;  // transition accumulators behind tot_frames (num_tids + 1 entries, 0 = none)
  vb::DevBuf d_acc;  // [occ N | mean N*D | var N*D | tot_like | tot_frames | transition accs]
  vb::DevBuf d_feats, d_feats2, d_ids, d_w;
  vb::DevBuf d_work;  // counting-sort workspace of the bucketed accumulation (accum.cu)
  bool bucket_attr_set = false;
};

struct vbgpu_lda_s {
  vb::StreamOrder order;  // cross-stream ordering of the handle's scratch (see StreamOrder)
  int device = 0;
  vb::Stream stream;
  int32_t C = 0, D = 0;
  int64_t n_doubles = 0;  // C + C*D + D(D+1)/2
  vb::DevBuf d_acc;       // [zero C | first C*D | second D(D+1)/2, SpMatrix packing]
  vb::DevBuf d_bad;       // uint64 count of invalid class ids since the last query
  vb::DevBuf d_work;      // counting-sort workspace
  vb::DevBuf d_feats, d_ids, d_w;  // staging of the host entry point
};

struct vbgpu_tree_s {
  vb::StreamOrder order;  // cross-stream ordering of the handle's scratch (see StreamOrder)
  int device = 0;
  vb::Stream stream;
  int32_t N = 3, P = 1, D = 0, max_keys = 0, num_tids = 0;
  uint32_t mask = 0;                 // hash table slots - 1 (a power of two >= 2 max_keys)
  vb::DevBuf d_info, d_ts;           // per transition-id: packed phone / pdf-class / flags, transition state
  vb::DevBuf d_acc;                  // [count K | sum_x K*D | sum_x2 K*D], K = max_keys, by dense id
  vb::DevBuf d_hkeys, d_hvals, d_keys_by_id;  // hash table (open addressing on the 64-bit key) and key of each dense id
  vb::DevBuf d_ctr;                  // uint64 counters (tree.cu)
  vb::DevBuf d_seg, d_seg_phone, d_ids, d_work;  // per-frame scratch and the counting-sort workspace
  vb::DevBuf d_feats, d_tids, d_stage;           // staging of the host entry points
  vb::BatchLayout layout;
};

struct vbgpu_pipeline_s {
  vb::StreamOrder order;  // cross-stream ordering of the handle's scratch (see StreamOrder)
  vbgpu_mfcc_t mfcc = nullptr;
  vbgpu_feat_t feat = nullptr;
  vbgpu_gmm_t gmm = nullptr;
  int device = 0;
  vb::Stream stream, copy_stream;
  vb::DevBuf d_mfcc, d_feats, d_pcm, d_ll[2], d_fmllr, d_stats;
  vb::PinBuf pin_pcm, pin_ll[2], pin_feats;
  vb::Event ev_ll[2], ev_copied[2];
};

// ---- kernel launchers (defined in the .cu files) ----------------------------------------------------------------
namespace vb {

int mfcc_build_tables(vbgpu_mfcc_t h);
int mfcc_launch(vbgpu_mfcc_t h, const void *d_pcm, bool is_f32, float *d_out, int32_t out_stride, cudaStream_t s);

int feat_compute_norm(vbgpu_feat_t h, const double *d_stats, int32_t n_spk, cudaStream_t s);
int feat_launch_stats(vbgpu_feat_t h, const float *d_feats, int32_t stride, double *d_stats, int32_t n_spk,
                      cudaStream_t s);
int feat_launch(vbgpu_feat_t h, const float *d_in, int32_t in_stride, const float *d_fmllr, int32_t fmllr_cols,
                float *d_out, int32_t out_stride, cudaStream_t s);

int score_simt_launch(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, float *d_ll, int32_t ll_stride,
                      cudaStream_t s);
int acc_posterior_ab_launch(vbgpu_gmm_t g, DevBuf *work, const float *d_feats, int64_t T, int32_t stride,
                            const int32_t *d_ids, const float *d_w, float *d_ab, int32_t ab_pitch, float *d_cnt,
                            double *d_like, int32_t *max_gauss_served, cudaStream_t s);
int score_tc_prepare(vbgpu_gmm_t h, const float *gconsts, const float *miv, const float *iv, int32_t stride);
bool score_tc_available(vbgpu_gmm_t h);
// native != 0: d_ll in device column order ([T x ll_stride], ll_stride >= score_tc_num_cols()); 0: the model's pdf order
int score_tc_launch(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, float *d_ll, int32_t ll_stride,
                    int native, cudaStream_t s);
int score_tc_rescored(vbgpu_gmm_t h, int64_t *n);        // frames of the last launch re-scored in FP32
int32_t score_tc_num_cols(vbgpu_gmm_t h);                 // P when the model is not on the tensor-core plan
const int32_t *score_tc_col_of_pdf(vbgpu_gmm_t h);        // host [P], null = identity
const int32_t *score_tc_col_of_pdf_dev(vbgpu_gmm_t h);    // device [P], null = identity
void score_tc_release(vbgpu_gmm_t h);
int score_tc_update_gconsts(vbgpu_gmm_t h, const float *gconsts);
int score_tc_debug_layout(int32_t P, int32_t D, const int32_t *pdf_offsets, const float *gconsts, const float *miv,
                          const float *iv, int32_t stride, int32_t pair, int32_t *info, uint8_t *image, int64_t image_cap,
                          int32_t *hdr, int32_t hdr_cap, int32_t *grp, int32_t grp_cap, int32_t *col_of_pdf, int32_t *merge,
                          int32_t merge_cap, float *centre, float *s1, float *s2, int32_t *bounds);

int sparse_subset_launch(const float *d_slab, int32_t slab_stride, int64_t t0, int64_t t1, const int32_t *d_frame2utt,
                         const int64_t *d_frame_offsets, const int64_t *d_sub_offsets, const int32_t *d_cols,
                         const int64_t *d_out_offsets, float *d_out, cudaStream_t s);
int sparse_gather_launch(const float *d_slab, int32_t slab_stride, int64_t t0, int64_t t1, const int32_t *d_frames,
                         const int32_t *d_cols, int64_t n, float *d_out, cudaStream_t s);

// Counting sort of T frames by bin id (pdf or class) in [0, P): ids outside go to bin P, which gets no work units, and
// are added to *bad.  Bin p then owns order[start[p] .. start[p+1]) and work units [unit_off[p], unit_off[p+1]) of up to
// kSortChunk frames each; unit_off[P+1] is the total.  With d_pdf_offsets, only pdfs of at most 64 Gaussians get units
// (the bucketed EM kernel's limit); NULL gives every bin its units.  work is the caller's (grown as needed).
constexpr int kSortChunk = 128;
struct BinSort {
  const int32_t *start, *unit_off, *order;
};
int bin_sort_launch(const int32_t *d_ids, int64_t T, int32_t P, const int32_t *d_pdf_offsets, int device, DevBuf *work,
                    unsigned long long *bad, cudaStream_t s, BinSort *out);

int lda_launch(vbgpu_lda_t h, const float *d_feats, int64_t T, int32_t stride, const int32_t *d_ids, const float *d_w,
               cudaStream_t s);

int tree_check(const vbgpu_tree_opts *o, const vbgpu_tid_tables *t, int32_t dim, int32_t max_keys);
int tree_init(vbgpu_tree_t h, const vbgpu_tree_opts *o, const vbgpu_tid_tables *t);  // h->D, max_keys, stream set
int tree_zero(vbgpu_tree_t h, cudaStream_t s);
int tree_launch(vbgpu_tree_t h, const float *d_feats, int32_t stride, const int32_t *d_tids, const int64_t *d_fo,
                int32_t n_utts, int64_t T, cudaStream_t s);
int tree_counters(vbgpu_tree_t h, int64_t *bad_utts, int64_t *dropped, int64_t *num_keys, bool reset);
int tree_download(vbgpu_tree_t h, int32_t *pdf_class, int32_t *phones, double *count, double *sum_x, double *sum_x2);
int tree_add(vbgpu_tree_t h, int32_t n, const int32_t *pdf_class, const int32_t *phones, const double *count,
             const double *sum_x, const double *sum_x2, int64_t *dropped);

int acc_launch(vbgpu_acc_t h, const float *d_feats, const float *d_feats2, int64_t T, int32_t stride,
               const int32_t *d_ids, const float *d_w, cudaStream_t s);
int acc_axpy(double *d_dst, const double *d_src, double scale, int64_t n, cudaStream_t s);
int acc_transitions_launch(double *d_trans, int32_t n_trans, const int32_t *d_tids, int64_t T, unsigned long long *bad,
                           cudaStream_t s);

}  // namespace vb
