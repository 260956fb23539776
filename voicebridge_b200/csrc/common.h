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

// The error count of one host-form call, in a slot of its own: the call neither reads nor resets the running count that
// the _dev calls add to (vbgpu_gmm_bad_count), and errors of other calls never show up in it.  begin() zeroes the slot on
// s and hands out its device pointer; end() copies it back and synchronises s.  Host forms run on their handle's own
// stream and synchronise before they return, so the slot needs no StreamOrder.
struct CallCount {
  DevBuf slot;
  int begin(cudaStream_t s, unsigned long long **bad) {
    VB_TRY(slot.reserve(8));
    VB_CUDA(cudaMemsetAsync(slot.p, 0, 8, s));
    *bad = slot.as<unsigned long long>();
    return 0;
  }
  int end(cudaStream_t s, unsigned long long *n) {
    VB_CUDA(cudaMemcpyAsync(n, slot.p, 8, cudaMemcpyDeviceToHost, s));
    VB_CUDA(cudaStreamSynchronize(s));
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
  vb::DevBuf d_bad;                             // uint64 running count of the _dev calls' errors (vbgpu_gmm_bad_count)
  vb::CallCount count;                          // the host forms' own errors
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
  vb::CallCount count;  // the host forms' own errors (the _dev forms count into the model's running count)
  bool bucket_attr_set = false;
};

struct vbgpu_lda_s {
  vb::StreamOrder order;  // cross-stream ordering of the handle's scratch (see StreamOrder)
  int device = 0;
  vb::Stream stream;
  int32_t C = 0, D = 0;
  int64_t n_doubles = 0;  // C + C*D + D(D+1)/2
  vb::DevBuf d_acc;       // [zero C | first C*D | second D(D+1)/2, SpMatrix packing]
  vb::DevBuf d_bad;       // uint64 count of invalid class ids of the _dev calls since the last query
  vb::CallCount count;    // the host entry point's own invalid class ids
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

namespace vb {
// Forced alignment (align.cu).  Graph limits: the costs of a CTA's states and its staged rows live in shared memory.
constexpr int32_t kAlignMaxStates = 4096, kAlignMaxSubset = 8192;
constexpr int64_t kAlignDefaultWorkspace = 4ll << 30;  // traceback entries + subset log-likelihoods of one group
struct AlignUtt {  // per utterance, fixed at create
  int32_t S, start, n_sub, n_lvls;
  int32_t state_base;  // first final cost
  int32_t csr_base;    // first of the S + 1 offsets of its emitting / epsilon incoming-arc lists
  int32_t lvl_base;    // first of its n_lvls + 1 level offsets
  int32_t arc_base;    // first of its arcs in the original order
};
struct AlignCall {  // per utterance and call
  int64_t f0, T;    // first row of the batch, frames
  int64_t ll_off;   // its [T x n_sub] block in the group's subset log-likelihoods
  int64_t tb_off;   // its [(T + 1) x S] traceback entries in the group's workspace
};
}  // namespace vb

struct vbgpu_align_s {
  vb::StreamOrder order;  // cross-stream ordering of the handle's scratch (see StreamOrder)
  int device = 0;
  vb::Stream stream;
  int32_t n_utts = 0, num_tids = 0, max_pdf = -1;
  int64_t n_arcs = 0;
  int32_t tb_bytes = 2;  // traceback entry: int16 when every utterance has fewer than 32768 arcs, else int32
  int64_t workspace_cap = vb::kAlignDefaultWorkspace;
  std::vector<int32_t> h_S, h_nsub;   // states and subset size per utterance
  std::vector<int64_t> h_sub_off;     // pdf subsets (what the subset scorer is asked for)
  std::vector<int32_t> h_sub_pdfs;
  vb::DevBuf d_utts, d_eoff, d_xoff, d_arcs, d_cw, d_clab, d_lvl_off, d_lvl_states, d_final, d_asrc, d_alab, d_tid2pdf;
  vb::DevBuf d_tid_cost, d_calls, d_best, d_ll, d_tb;  // per-call scratch
  vb::DevBuf d_feats, d_ali, d_pdf, d_tot;             // staging of the host form
  vb::CallCount count;                                 // the host form's own errors
};

namespace vb {
// Decoding (decode.cu).  The workspace of a group: per utterance vb::decode_ws_bytes, plus the log-likelihoods of the
// feature form.
constexpr int64_t kDecodeDefaultWorkspace = 16ll << 30;
struct DecodeCall {  // per utterance and call
  int64_t f0, T;     // first row of the batch, frames
  int64_t ll_row0;   // its first row in the log-likelihood matrix the search reads
  int64_t ws_off;    // its workspace, in bytes from the group's
  int64_t lat_off;   // lattice form: its lattice store (vb::lattice_arena_bytes), in bytes from the group's workspace
  int32_t NT, NL;    //   tokens and links the store holds
};
struct DecodeArgs {  // everything the search and traceback kernels read, for one group
  const DecodeCall *calls;
  unsigned char *ws;
  const int32_t *e_off, *x_off, *lvl;
  const int4 *e_arcs, *x_arcs;  // {dst, column (emitting) / -1, weight bits, original arc index}
  const float *finals, *ll;
  int64_t ll_stride;
  float scale, beam;
  int32_t max_active, S, start, n_lvls, cap, cap2, max_words;
  int32_t *best, *status, *ali, *pdf_ids, *words, *num_words;
  double *tot_cost;
  // lattice form
  float lattice_beam;
  int32_t max_states, max_arcs;
  const int32_t *ilabel, *olabel;  // by original arc index
  const float *weight;
  vbgpu_lattice_out lat;
};
}  // namespace vb

struct vbgpu_decoder_s {
  vb::StreamOrder order;  // cross-stream ordering of the handle's scratch (see StreamOrder)
  int device = 0;
  vb::Stream stream;
  int32_t S = 0, start = 0, num_tids = 0, max_pdf = -1, n_lvls = 0;
  int64_t n_emit = 0;  // emitting arcs
  int64_t workspace_cap = vb::kDecodeDefaultWorkspace;
  vb::DevBuf d_e_off, d_x_off, d_e_arcs, d_x_arcs, d_e_pdf, d_lvl, d_final, d_tid2pdf, d_ilabel, d_olabel, d_weight;
  vb::DevBuf d_calls, d_best, d_ws, d_ll;              // per-call scratch
  vb::DevBuf d_feats, d_ali, d_pdf, d_words, d_nw, d_tot, d_status;  // staging of the host forms
  vb::DevBuf d_lat[9], d_lat_n;                                     //   (lattice arrays; counts and status)
  vb::CallCount count;                                 // the host form's own errors
};

struct vbgpu_pipeline_s {
  vb::StreamOrder order;  // cross-stream ordering of the handle's scratch (see StreamOrder)
  vbgpu_mfcc_t mfcc = nullptr;
  vbgpu_feat_t feat = nullptr;
  vbgpu_gmm_t gmm = nullptr;
  int device = 0;
  vb::Stream stream, copy_stream;
  vb::DevBuf d_mfcc, d_feats, d_pcm, d_ll[2], d_fmllr, d_stats;
  vb::PinBuf pin_pcm, pin_ll[2];
  vb::Event ev_ll[2], ev_copied[2];
  vb::CallCount count;  // the host forms' own errors (the _dev forms count into the model's running count)
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

// The launchers that count errors (NaN/Inf results, invalid ids) add them to *bad: the caller decides which count that is.
int score_simt_launch(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, float *d_ll, int32_t ll_stride,
                      unsigned long long *bad, cudaStream_t s);
int acc_posterior_ab_launch(vbgpu_gmm_t g, DevBuf *work, const float *d_feats, int64_t T, int32_t stride,
                            const int32_t *d_ids, const float *d_w, float *d_ab, int32_t ab_pitch, float *d_cnt,
                            double *d_like, int32_t *max_gauss_served, unsigned long long *bad, cudaStream_t s);
int score_tc_prepare(vbgpu_gmm_t h, const float *gconsts, const float *miv, const float *iv, int32_t stride);
bool score_tc_available(vbgpu_gmm_t h);
// native != 0: d_ll in device column order ([T x ll_stride], ll_stride >= score_tc_num_cols()); 0: the model's pdf order
int score_tc_launch(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, float *d_ll, int32_t ll_stride,
                    int native, unsigned long long *bad, cudaStream_t s);
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
               unsigned long long *bad, cudaStream_t s);

int tree_check(const vbgpu_tree_opts *o, const vbgpu_tid_tables *t, int32_t dim, int32_t max_keys);
int tree_init(vbgpu_tree_t h, const vbgpu_tree_opts *o, const vbgpu_tid_tables *t);  // h->D, max_keys, stream set
int tree_zero(vbgpu_tree_t h, cudaStream_t s);
int tree_launch(vbgpu_tree_t h, const float *d_feats, int32_t stride, const int32_t *d_tids, const int64_t *d_fo,
                int32_t n_utts, int64_t T, cudaStream_t s);
int tree_counters(vbgpu_tree_t h, int64_t *bad_utts, int64_t *dropped, int64_t *num_keys, bool reset);
int tree_download(vbgpu_tree_t h, int32_t *pdf_class, int32_t *phones, double *count, double *sum_x, double *sum_x2);
int tree_add(vbgpu_tree_t h, int32_t n, const int32_t *pdf_class, const int32_t *phones, const double *count,
             const double *sum_x, const double *sum_x2, int64_t *dropped);

int align_create(int32_t n_utts, const int32_t *state_offsets, const int32_t *start, const float *final_cost,
                 const int64_t *arc_offsets, const int32_t *arc_src, const int32_t *arc_dst, const int32_t *arc_ilabel,
                 const float *arc_weight, const int32_t *tid2pdf, int32_t num_tids, int device, vbgpu_align_t *out);
int align_set_weights(vbgpu_align_t h, const float *tid_cost, cudaStream_t s);  // this call's arc weights
// Utterances [u0, u0 + n) of a group: d_ll their subset blocks, d_tb their traceback workspace (AlignCall offsets).
int align_group_launch(vbgpu_align_t h, int32_t u0, int32_t n, int32_t max_S, int32_t max_sub, const float *d_ll,
                       float acoustic_scale, void *d_tb, int32_t *d_ali, int32_t *d_pdf_ids, double *d_tot_cost,
                       cudaStream_t s);

int decoder_create(int32_t num_states, int32_t start, const float *final_cost, int64_t num_arcs, const int32_t *arc_src,
                   const int32_t *arc_dst, const int32_t *arc_ilabel, const int32_t *arc_olabel, const float *arc_weight,
                   const int32_t *tid2pdf, int32_t num_tids, int device, vbgpu_decoder_t *out);
// Workspace bytes of one utterance: T frames, cap tokens per set, cap2 survivor records per frame.
int64_t decode_ws_bytes(int32_t S, int32_t cap, int32_t cap2, int32_t n_lvls, int64_t T);
int decoder_set_cols(vbgpu_decoder_t h, const int32_t *d_col_of_pdf, cudaStream_t s);  // null map: identity
int decoder_count_bad(const float *d_ll, int32_t ll_stride, int64_t T, const int32_t *d_col_of_pdf, int32_t P,
                      unsigned long long *bad, cudaStream_t s);
// Lattice store bytes of one utterance: NT tokens, NL links, T frames.
int64_t lattice_arena_bytes(int32_t NT, int32_t NL, int32_t cap, int32_t cap2, int64_t T);
int decoder_search_launch(const DecodeArgs &a, int32_t u0, int32_t n, bool lattice, cudaStream_t s);
int decoder_lattice_launch(const DecodeArgs &a, int32_t u0, int32_t n, cudaStream_t s);
int decoder_traceback_launch(vbgpu_decoder_t h, const DecodeArgs &a, int32_t u0, int32_t n, cudaStream_t s);

int acc_launch(vbgpu_acc_t h, const float *d_feats, const float *d_feats2, int64_t T, int32_t stride,
               const int32_t *d_ids, const float *d_w, unsigned long long *bad, cudaStream_t s);
int acc_axpy(double *d_dst, const double *d_src, double scale, int64_t n, cudaStream_t s);
int acc_transitions_launch(double *d_trans, int32_t n_trans, const int32_t *d_tids, int64_t T, unsigned long long *bad,
                           cudaStream_t s);

}  // namespace vb
