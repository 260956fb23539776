/* vbgpu.h — C ABI of libvbgpu.so: the B200 (sm_100a) implementation of VoiceBridge's acoustic-scoring
 * hot path  PCM -> MFCC -> CMVN / delta | splice+LDA / fMLLR -> diag-GMM log-likelihoods | EM statistics.
 *
 * This is the drop-in boundary.  The reference has no FFI; its seams for this path are C++ types of the
 * Kaldi snapshot linked into the VoiceBridge DLL (paths relative to /root/reference/kaldi-master/src,
 * VB = /root/reference/VoiceBridge/VoiceBridge/kaldi-win):
 *
 *   vbgpu_wave_*      replaces  WaveData::Read                                      feat/wave-reader.cc:119-310
 *                               (caller VB/src/featbin/compute-mfcc-feats.cpp:110-135)
 *   vbgpu_downsample_* replaces DownsampleWaveForm (the allow_downsample branch of ComputeFeatures)   feat/resample.cc:368-376,
 *                               feat/feature-common-inl.h:37-48
 *   vbgpu_mfcc_*      replaces  OfflineFeatureTpl<MfccComputer>::ComputeFeatures   feat/feature-common.h:110-178,
 *                               feat/feature-common-inl.h:29-98 (caller VB/src/featbin/compute-mfcc-feats.cpp:147)
 *   vbgpu_cmvn_stats  replaces  AccCmvnStats                                       transform/cmvn.cc:30-62
 *                               (caller VB/src/featbin/compute-cmvn-stats.cpp)
 *   vbgpu_feat_*      replaces  ApplyCmvn + ComputeDeltas | SpliceFrames + transform-feats GEMM (+ per-speaker fMLLR)
 *                               transform/cmvn.cc:64-113, feat/feature-functions.cc:160-171,205-226,
 *                               VB/src/featbin/transform-feats.cpp:95-107 (callers VB/scr/steps/decode_gmm.cpp:395-571)
 *   vbgpu_gmm_*       replaces  AmDiagGmm / DiagGmm::LogLikelihoods + LogSumExp behind DecodableAmDiagGmmScaled
 *                               gmm/diag-gmm.cc:528-562, gmm/decodable-am-diag-gmm.cc:28-72, matrix/kaldi-vector.cc:757-775
 *                               (callers decoder/lattice-faster-decoder.cc:727,754, decoder/faster-decoder.cc:250,276)
 *   vbgpu_acc_*       replaces  AccumAmDiagGmm::AccumulateForGmm[Twofeats] / AccumDiagGmm   gmm/mle-am-diag-gmm.cc:69-97,
 *                               gmm/mle-diag-gmm.cc:171-204 (caller VB/src/gmmbin/gmm-acc-stats-ali.cpp:89-94) and the
 *                               file-based reduce of VB/src/gmmbin/gmm-sum-accs.cpp:44-50 (vbgpu_acc_add / all-reduce)
 *   vbgpu_fmllr_*     replaces  FmllrDiagGmmAccs::AccumulateForGmm (fMLLR statistics beta, K, G per speaker)
 *                               transform/fmllr-diag-gmm.cc:30-45,110-121,562-583 (caller VB/src/gmmbin/gmm-est-fmllr.cpp:40-55)
 *   vbgpu_lda_*       replaces  LdaEstimate::Init / ZeroAccumulators / Accumulate (LDA class statistics of acc-lda)
 *                               transform/lda-estimate.{h,cc} (caller VB/scr/steps/train_lda_mllt.cpp) and the summing of
 *                               the per-job lda.*.acc files by est-lda (vbgpu_lda_allreduce)
 *   vbgpu_tree_*      replaces  AccumulateTreeStats (tree statistics of acc-tree-stats, with SplitToPhones / IsReordered)
 *                               hmm/tree-accu.cc, hmm/hmm-utils.cc, tree/clusterable-classes.cc (callers train_deltas,
 *                               train_lda_mllt, train_sat) and the summing of the per-job treeacc files (sum-tree-stats)
 *   vbgpu_io_*        reads / writes  Matrix / CompressedMatrix / Vector / int32-vector objects, archive entries, model
 *                               files (-> tid2pdf + flattened AmDiagGmm) and gmm-acc-stats-ali statistics files
 *                               matrix/kaldi-matrix.cc:1375-1460, matrix/compressed-matrix.cc:531-670, gmm/diag-gmm.cc:705-756
 *   vbgpu_pitch_*     replaces  ComputeKaldiPitch / ProcessPitch / ComputeAndProcessKaldiPitch (offline mode)
 *                               feat/pitch-functions.cc:1291-1325,1581-1665, feat/resample.cc:34-309
 *                               (callers VB/src/featbin/compute-kaldi-pitch-feats.cpp:95, process-kaldi-pitch-feats.cpp:76)
 *   vbgpu_pipeline_*  the fused measured path PCM -> loglikes (MFCC, feature pipeline and scoring in one call)
 *
 * Conventions
 *   - Every function returns int: 0 = ok, <0 = error (VBGPU_ERR_*); no exception crosses the boundary (the reference's
 *     L3 functions return -1 on KALDI_ERR, compute-mfcc-feats.cpp:192-197).  vbgpu_last_error() gives the text of
 *     the calling thread's last error.
 *   - Matrices follow kaldi::Matrix<BaseFloat> (matrix/kaldi-matrix.h:61-117): row-major float, explicit row stride in
 *     floats (Kaldi's own stride is cols rounded up to 4).  The caller owns host memory; the library owns device memory.
 *   - Utterances are batched: utterance u owns samples [sample_offsets[u], sample_offsets[u+1]) of one packed PCM
 *     array and rows [frame_offsets[u], frame_offsets[u+1]) of every packed feature / log-likelihood matrix.
 *   - pdf-ids are 0-based, frames 0-based (transition-id -> pdf-id mapping stays on the host, hmm/transition-model.h:324).
 *   - Functions with suffix _dev take DEVICE pointers and a cudaStream_t (passed as void*); they enqueue work and return
 *     without synchronising.  All other functions take HOST pointers and are synchronous.
 *   - A handle is bound to one CUDA device and owns one stream; handles are not thread-safe, the library is (different
 *     handles may be used concurrently from the nj host threads of VB/scr/steps/ sources).  _dev calls on one handle may
 *     use different streams from call to call: the handle's scratch (batch layouts, statistics, work space) is ordered
 *     across streams by an event (a call on a new stream waits for the previous call), the caller's own buffers are not.
 *   - There is NO CPU fallback: without a CUDA device every create call fails with VBGPU_ERR_CUDA.
 */
#ifndef VBGPU_H_
#define VBGPU_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VBGPU_OK 0
#define VBGPU_ERR_INVALID (-1) /* bad argument / dimension mismatch (KALDI_ERR in the reference) */
#define VBGPU_ERR_CUDA (-2)    /* CUDA runtime failure, or no device */
#define VBGPU_ERR_NUMERIC (-3) /* NaN/Inf log-likelihood (decodable-am-diag-gmm.cc:65-66), count<1 in CMVN ... */
#define VBGPU_ERR_NOMEM (-4)

/* Mirror of MfccOptions + FrameExtractionOptions + MelBanksOptions
 * (feat/feature-mfcc.h:38-78, feat/feature-window.h:35-101, feat/mel-computations.h:43-74). */
typedef struct vbgpu_mfcc_opts {
  float samp_freq;               /* 16000 */
  float frame_shift_ms;          /* 10 */
  float frame_length_ms;         /* 25 */
  float dither;                  /* Kaldi default 1.0.  !=0 uses a counter-based generator, not libc rand() */
  float preemph_coeff;           /* 0.97 */
  int32_t remove_dc_offset;      /* 1 */
  int32_t window_type;           /* 0 povey, 1 hamming, 2 hanning, 3 rectangular, 4 blackman */
  int32_t round_to_power_of_two; /* 1 (0 is rejected: only the split-radix branch, feature-mfcc.cc:41-42, is built) */
  float blackman_coeff;          /* 0.42 */
  int32_t snip_edges;            /* 1 */
  int32_t num_bins;              /* 23 (<= 32) */
  float low_freq;                /* 20 */
  float high_freq;               /* 0 */
  float vtln_low;                /* 100 */
  float vtln_high;               /* -500 */
  int32_t htk_mode;              /* 0 */
  int32_t num_ceps;              /* 13 (<= num_bins) */
  int32_t use_energy;            /* Kaldi default 1; the recipes use 0 */
  float energy_floor;            /* 0 */
  int32_t raw_energy;            /* 1 */
  float cepstral_lifter;         /* 22 */
  int32_t htk_compat;            /* 0 */
} vbgpu_mfcc_opts;

/* Feature post-processing options: apply-cmvn (--norm-means/--norm-vars, apply-cmvn.cpp:30-60), then either
 * add-deltas (DeltaFeaturesOptions, feat/feature-functions.h:50-61) or splice-feats + transform-feats. */
typedef struct vbgpu_feat_opts {
  int32_t norm_means;   /* 1 */
  int32_t norm_vars;    /* 0 */
  int32_t mode;         /* 0 = "delta": CMVN -> deltas;  1 = "lda": CMVN -> splice -> matrix (decode_gmm.cpp:103-105) */
  int32_t delta_order;  /* 2 */
  int32_t delta_window; /* 2 */
  int32_t splice_left;  /* 3 (splice-feats default is 4, splice-feats.cpp:30) */
  int32_t splice_right; /* 3 */
} vbgpu_feat_opts;

typedef struct vbgpu_mfcc_s *vbgpu_mfcc_t;
typedef struct vbgpu_feat_s *vbgpu_feat_t;
typedef struct vbgpu_gmm_s *vbgpu_gmm_t;
typedef struct vbgpu_acc_s *vbgpu_acc_t;
typedef struct vbgpu_fmllr_s *vbgpu_fmllr_t;
typedef struct vbgpu_pipeline_s *vbgpu_pipeline_t;
typedef struct vbgpu_pitch_s *vbgpu_pitch_t;
typedef struct vbgpu_lda_s *vbgpu_lda_t;
typedef struct vbgpu_tree_s *vbgpu_tree_t;

/* ---- library ------------------------------------------------------------------------------------------------ */
int vbgpu_version(void);
const char *vbgpu_last_error(void);
int vbgpu_device_count(int *count);

/* ---- WAV container (host-side I/O in front of the path) -------------------------------------------------------- */
/* WaveInfo::Read / WaveData::Read (feat/wave-reader.cc:119-310) on an in-memory RIFF/RIFX image: 16-bit PCM or
 * WAVE_FORMAT_EXTENSIBLE/PCM, extra chunks skipped, "stream mode" sizes and truncated data accepted as the reference does.
 * Byte handling only, no device work; samples stay int16 (the reference keeps the int16 range, wave-reader.cc:302-309). */
typedef struct vbgpu_wave_info {
  float samp_freq;
  int32_t num_channels;
  int64_t num_samples; /* per channel */
  int64_t data_offset; /* byte offset of the first sample in the image */
  int32_t reverse_bytes; /* RIFX */
} vbgpu_wave_info;
int vbgpu_wave_parse(const void *bytes, size_t n_bytes, vbgpu_wave_info *info);
/* One channel, de-interleaved, host byte order: out[num_samples].  channel < 0 = first channel
 * (compute-mfcc-feats --channel=-1, compute-mfcc-feats.cpp:120-135). */
int vbgpu_wave_channel_i16(const void *bytes, size_t n_bytes, const vbgpu_wave_info *info, int32_t channel, int16_t *out);

/* DownsampleWaveForm (feat/resample.cc:368-376) — the one thing OfflineFeatureTpl::ComputeFeatures does besides Compute: a wave
 * whose sampling rate is ABOVE the options' is low-pass filtered and resampled (LinearResample, cutoff 0.99 * new_freq / 2,
 * 6 zeros, one flushed call) when --allow-downsample is set; a rate below is always an error (feature-common-inl.h:29-55).
 * A handle holds the filter tables of one (orig_freq, new_freq) pair.  num_out = LinearResample::GetNumOutputSamples(n, true). */
typedef struct vbgpu_resample_s *vbgpu_resample_t;
int vbgpu_downsample_create(float orig_freq, float new_freq, int32_t device, vbgpu_resample_t *out);
void vbgpu_downsample_destroy(vbgpu_resample_t h);
int64_t vbgpu_downsample_num_out(vbgpu_resample_t h, int64_t n_in);
int vbgpu_downsample_f32(vbgpu_resample_t h, const float *wave, int64_t n_in, float *out /* num_out floats, host */);
int vbgpu_downsample_dev(vbgpu_resample_t h, const float *d_wave, int64_t n_in, float *d_out, void *stream);

/* ---- MFCC front end ------------------------------------------------------------------------------------------- */
void vbgpu_mfcc_opts_default(vbgpu_mfcc_opts *opts);
int vbgpu_mfcc_create(const vbgpu_mfcc_opts *opts, int device, vbgpu_mfcc_t *out);
/* OfflineFeatureTpl<FbankComputer> (feat/feature-fbank.cc:73-123, SURVEY.md §8f n4): the same handle type and compute
 * entry points, with the filterbank tail instead of the DCT.  Frame, mel, energy and htk_compat options are taken from
 * opts (num_ceps, cepstral_lifter unused); output = num_bins columns, +1 with use_energy (first, or last with htk_compat). */
int vbgpu_fbank_create(const vbgpu_mfcc_opts *opts, int32_t use_log_fbank, int32_t use_power, int device,
                       vbgpu_mfcc_t *out);
/* OfflineFeatureTpl<PlpComputer> (feat/feature-plp.cc:25-188, mel-computations.cc:269-340): equal-loudness, cube-root
 * compression, cosine IDFT to an autocorrelation, Levinson-Durbin, LPC -> cepstrum.  num_ceps columns (C0 = residual
 * log-energy, or the frame log-energy with use_energy); num_ceps <= lpc_order + 1 <= 31, num_bins <= 30. */
int vbgpu_plp_create(const vbgpu_mfcc_opts *opts, int32_t lpc_order, float compress_factor, float cepstral_scale,
                     int device, vbgpu_mfcc_t *out);
int vbgpu_mfcc_destroy(vbgpu_mfcc_t h);
int vbgpu_mfcc_dim(vbgpu_mfcc_t h);                              /* MfccComputer::Dim() = num_ceps */
int64_t vbgpu_mfcc_num_frames(vbgpu_mfcc_t h, int64_t n_samples); /* NumFrames(), feature-window.cc:41-87 */
/* Fills frame_offsets[n_utts+1] from sample_offsets[n_utts+1]; returns total frames or <0. */
int64_t vbgpu_mfcc_frame_offsets(vbgpu_mfcc_t h, const int64_t *sample_offsets, int32_t n_utts, int64_t *frame_offsets);
/* Batched ComputeFeatures.  pcm: int16 samples as WaveData holds them (NOT scaled to +-1, wave-reader.cc:302-309);
 * the _f32 form takes the float copies Kaldi's API takes.  vtln_warp: per-utterance factors or NULL (=1.0).
 * out: [total_frames x out_stride] floats, cols = num_ceps. */
int vbgpu_mfcc_compute_i16(vbgpu_mfcc_t h, const int16_t *pcm, const int64_t *sample_offsets, int32_t n_utts,
                           const float *vtln_warp, float *out, int32_t out_stride);
int vbgpu_mfcc_compute_f32(vbgpu_mfcc_t h, const float *wave, const int64_t *sample_offsets, int32_t n_utts,
                           const float *vtln_warp, float *out, int32_t out_stride);
/* Device form: d_pcm device pointer (int16 if is_f32==0), offsets on the HOST; d_out device [frames x out_stride]. */
int vbgpu_mfcc_compute_dev(vbgpu_mfcc_t h, const void *d_pcm, int32_t is_f32, const int64_t *sample_offsets,
                           int32_t n_utts, const float *vtln_warp, float *d_out, int32_t out_stride, void *stream);

/* ---- CMVN statistics + feature pipeline ---------------------------------------------------------------------------- */
void vbgpu_feat_opts_default(vbgpu_feat_opts *opts);
/* transform: the global LDA/MLLT matrix `final.mat` [rows x cols], cols == spliced dim or spliced dim + 1
 * (transform-feats.cpp:95-107); must be NULL in delta mode. in_dim = MFCC dim. */
int vbgpu_feat_create(const vbgpu_feat_opts *opts, int32_t in_dim, const float *transform, int32_t rows, int32_t cols,
                      int device, vbgpu_feat_t *out);
int vbgpu_feat_destroy(vbgpu_feat_t h);
int vbgpu_feat_out_dim(vbgpu_feat_t h);
/* AccCmvnStats per speaker: stats[n_spk][2][dim+1] doubles are ADDED to (compute-cmvn-stats.cpp).
 * utt2spk[u] in [0,n_spk) or NULL (per-utterance stats, n_spk == n_utts). */
int vbgpu_cmvn_stats(vbgpu_feat_t h, const float *feats, int32_t stride, const int64_t *frame_offsets, int32_t n_utts,
                     const int32_t *utt2spk, int32_t n_spk, double *stats);
/* apply-cmvn | add-deltas  or  apply-cmvn | splice-feats | transform-feats, then optional per-speaker fMLLR
 * (fmllr[n_spk][out_dim][out_dim+1] or [out_dim][out_dim], selected by fmllr_cols; NULL = none).
 * cmvn_stats may be NULL only if norm_means == norm_vars == 0. */
int vbgpu_feat_run(vbgpu_feat_t h, const float *feats, int32_t in_stride, const int64_t *frame_offsets, int32_t n_utts,
                   const int32_t *utt2spk, int32_t n_spk, const double *cmvn_stats, const float *fmllr,
                   int32_t fmllr_cols, float *out, int32_t out_stride);
/* Device form of vbgpu_feat_run: d_feats, d_out and d_fmllr are device pointers; frame_offsets, utt2spk and cmvn_stats stay
 * host arrays.  Speakers with a CMVN count below 1 (or non-finite statistics) are rejected on the host before any work.
 * Splice-only output (what acc-lda reads): lda mode with the K x K identity as transform (K = in_dim * (left + right + 1))
 * gives the spliced CMVN'd rows bit for bit, since the kernel's products with 1 and 0 are exact.  The transform has to fit
 * the kernel's shared memory (K = 91 and 117 do; larger K fails cleanly at launch) and costs K^2 FP32 multiply-adds per
 * frame. */
int vbgpu_feat_run_dev(vbgpu_feat_t h, const float *d_feats, int32_t in_stride, const int64_t *frame_offsets,
                       int32_t n_utts, const int32_t *utt2spk, int32_t n_spk, const double *cmvn_stats,
                       const float *d_fmllr, int32_t fmllr_cols, float *d_out, int32_t out_stride, void *stream);

/* ---- acoustic model + scoring ------------------------------------------------------------------------------------------ */
/* Flattened AmDiagGmm: pdf p owns Gaussians [pdf_offsets[p], pdf_offsets[p+1]); arrays are what
 * DiagGmm::gconsts()/means_invvars()/inv_vars() return (diag-gmm.h:174-180), rows packed with stride `stride`. */
int vbgpu_gmm_create(int32_t num_pdfs, int32_t dim, const int32_t *pdf_offsets, const float *gconsts,
                     const float *means_invvars, const float *inv_vars, int32_t stride, int device, vbgpu_gmm_t *out);
int vbgpu_gmm_destroy(vbgpu_gmm_t h);
int vbgpu_gmm_num_pdfs(vbgpu_gmm_t h);
int vbgpu_gmm_num_gauss(vbgpu_gmm_t h);
int vbgpu_gmm_dim(vbgpu_gmm_t h);
/* GmmBoostSilence-style update of gconsts only (gmm-boost-silence.cpp): new values for all N Gaussians. */
int vbgpu_gmm_set_gconsts(vbgpu_gmm_t h, const float *gconsts);
/* Select the scoring kernel: 0 = auto (tensor-core path when the model fits it), 1 = FP32 SIMT, 2 = tcgen05. */
int vbgpu_gmm_set_kernel(vbgpu_gmm_t h, int32_t kind);
/* Dense scoring: loglikes[t*ll_stride + p] = LogSumExp_m( gconst + means_invvars.x - 0.5 inv_vars.x^2 ), all pdfs,
 * all frames: the matrix DecodableAmDiagGmmUnmapped::LogLikelihoodZeroBased would fill lazily.
 * Returns VBGPU_ERR_NUMERIC if any value is NaN/Inf (the reference raises KALDI_ERR). */
int vbgpu_gmm_score(vbgpu_gmm_t h, const float *feats, int64_t T, int32_t stride, float *loglikes, int32_t ll_stride);
int vbgpu_gmm_score_dev(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, float *d_loglikes,
                        int32_t ll_stride, void *stream);
/* DEVICE COLUMN ORDER.  The tensor-core kernel lays the Gaussians out for its epilogue (pdfs sorted by size, 16 to a
 * group), so its natural output is a matrix whose column col_of_pdf[p] holds pdf p; it has vbgpu_gmm_num_cols() >= P
 * columns (padding members and the pieces of very large pdfs take columns too).  Every consumer of the matrix indexes it
 * through a map anyway (a decodable: frame, transition-id -> tid2pdf -> pdf, decodable-am-diag-gmm.h:66-70), so the
 * fast entry points below hand out that layout and the map; the pdf-order entry points above stay, at the price of one
 * extra gather kernel.  For a model scored by the FP32 SIMT kernel the map is the identity and num_cols == P. */
int vbgpu_gmm_num_cols(vbgpu_gmm_t h);
int vbgpu_gmm_col_of_pdf(vbgpu_gmm_t h, int32_t *col_of_pdf /* [num_pdfs] */);
/* "" when the model is scored on the tensor cores, else the reason it is not (also printed once to stderr at create time
 * unless VBGPU_QUIET is set): the FP32 SIMT kernel is ~25x slower. */
const char *vbgpu_gmm_plan_note(vbgpu_gmm_t h);
/* d_loglikes[t*ll_stride + col_of_pdf[p]], ll_stride >= vbgpu_gmm_num_cols(). */
int vbgpu_gmm_score_cols_dev(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, float *d_loglikes,
                             int32_t ll_stride, void *stream);
/* Test hook (host only, needs no device): the tensor-core layout of a model for the CTA-pair (pair != 0) or single-CTA
 * kernel — info[8] = {K steps, panels, columns, merge entries, image bytes / 16, groups, pair, 0}, the fp16 hi/lo B image,
 * the panel headers (4 int32 each), the group entries (2 int32 each), the column map, the merge list (main column, extra
 * column), the centring / scaling vectors and the unit cut table bounds[64][65] (panel ranges of a frame tile cut into
 * k = 1..64 units).  Buffers may be NULL (sizes come back in info).
 * tests/test_tc_layout.py decodes the image on the CPU and checks it against the oracle. */
int vbgpu_debug_tc_layout(int32_t num_pdfs, int32_t dim, const int32_t *pdf_offsets, const float *gconsts,
                          const float *means_invvars, const float *inv_vars, int32_t stride, int32_t pair, int32_t *info,
                          uint8_t *image, int64_t image_cap, int32_t *hdr, int32_t hdr_cap, int32_t *grp, int32_t grp_cap,
                          int32_t *col_of_pdf, int32_t *merge, int32_t merge_cap, float *centre, float *s1, float *s2, int32_t *bounds);
/* Bytes of device memory and of pinned host memory the library holds right now, over all handles and devices of the
 * process (scratch included).  Creating and destroying a handle leaves both where they were; tests use this to check
 * that nothing leaks.  Needs no GPU. */
int vbgpu_debug_live_bytes(int64_t *device_bytes, int64_t *pinned_bytes);
/* SPARSE CONSUMERS (SURVEY.md §8f n3).  The dense matrix is 4 P bytes per frame; its consumers read far less, and shipping
 * only that is what takes the host path off the PCIe line.  Both forms score on the device in slabs of frames (bounded
 * footprint) and extract what was asked for; *_dev forms take device feature / output pointers (descriptors on the host).
 *
 * Subsets — forced alignment reads only the pdfs of the utterance's own training graph
 * (VB/src/gmmbin/gmm-align-compiled.cpp:119-128 builds one decodable per utterance and AlignUtteranceWrapper walks that
 * graph): utterance u owns rows [frame_offsets[u], frame_offsets[u+1]) and asks for pdfs
 * subset_pdfs[subset_offsets[u] .. subset_offsets[u+1]) (any order); its block of `out` starts at float out_offsets[u]
 * (filled when not NULL: the running sum of rows x subset size) and is [rows x subset size] row-major in the order given. */
int vbgpu_gmm_score_subset(vbgpu_gmm_t h, const float *feats, int64_t T, int32_t stride, const int64_t *frame_offsets,
                           int32_t n_utts, const int64_t *subset_offsets, const int32_t *subset_pdfs, float *out,
                           int64_t *out_offsets);
int vbgpu_gmm_score_subset_dev(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, const int64_t *frame_offsets,
                               int32_t n_utts, const int64_t *subset_offsets, const int32_t *subset_pdfs, float *d_out,
                               int64_t *out_offsets, void *stream);
/* Arcs — lattice rescoring asks for one (frame, pdf) pair per arc (lat/lattice-functions.cc:1214-1360
 * RescoreCompactLatticeInternal / RescoreLattice): out[i] = loglike(frames[i], pdfs[i]), frames indexing the packed rows. */
int vbgpu_gmm_score_gather(vbgpu_gmm_t h, const float *feats, int64_t T, int32_t stride, const int32_t *frames,
                           const int32_t *pdfs, int64_t n, float *out);
int vbgpu_gmm_score_gather_dev(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, const int32_t *frames,
                               const int32_t *pdfs, int64_t n, float *d_out, void *stream);
/* Number of NaN/Inf values produced by _dev calls since the last query (synchronises the handle's work). */
int vbgpu_gmm_bad_count(vbgpu_gmm_t h, int64_t *count);
/* Frames of the handle's last scoring launch that the tensor-core path handed to the FP32 kernel: features outside the
 * fp16 scaling plan, or every score so low (below -27000 nats) that the padding columns of the layout would show through.
 * The results are the reference's either way; a large count means a slow launch and, usually, a broken utterance or
 * transform upstream.  Synchronises the device.  0 for models scored by the FP32 kernel throughout. */
int vbgpu_gmm_rescored_frames(vbgpu_gmm_t h, int64_t *count);

/* DiagGmm::ComponentPosteriors (gmm/diag-gmm.cc:601-615) of each frame's aligned pdf, scaled by weights[t] (NULL = 1.0):
 * what gmm-post-to-gpost (VB/src/gmmbin) writes as Gaussian-level posteriors.  post receives, frame after frame, the
 * posteriors of the Gaussians of pdf_ids[t] (sum over frames of that pdf's size floats); loglikes[T] (nullable) the frames'
 * log-likelihoods. */
int vbgpu_gmm_component_posteriors(vbgpu_gmm_t model, const float *feats, int64_t T, int32_t stride, const int32_t *pdf_ids,
                                   const float *weights, float *post, float *loglikes);

/* ---- EM sufficient statistics --------------------------------------------------------------------------------------- */
int vbgpu_acc_create(vbgpu_gmm_t model, vbgpu_acc_t *out); /* AccumAmDiagGmm::Init(model, kGmmAll) */
/* The same with the transition accumulators gmm-acc-stats-ali keeps beside the GMM statistics
 * (VB/src/gmmbin/gmm-acc-stats-ali.cpp:92 trans_model.Accumulate(1.0, tid, &transition_accs); gmm-sum-accs.cpp:48 sums both):
 * num_tids = TransitionModel::NumTransitionIds().  They live BEHIND tot_frames in the one buffer (num_tids + 1 doubles,
 * indexed by the 1-based transition-id), so the single all-reduce / vbgpu_acc_add covers them too. */
int vbgpu_acc_create_with_transitions(vbgpu_gmm_t model, int32_t num_tids, vbgpu_acc_t *out);
int vbgpu_acc_destroy(vbgpu_acc_t h);
int vbgpu_acc_zero(vbgpu_acc_t h);
/* transition_accs[tids[t]] += 1 for every frame of an alignment (transition-ids, not pdf-ids). */
int vbgpu_acc_accumulate_transitions(vbgpu_acc_t h, const int32_t *tids, int64_t T);
int vbgpu_acc_accumulate_transitions_dev(vbgpu_acc_t h, const int32_t *d_tids, int64_t T, void *stream);
int vbgpu_acc_download_transitions(vbgpu_acc_t h, double *trans_accs /* [num_tids + 1], entry 0 unused */);
/* AccumulateForGmm for every frame of an alignment: pdf_ids[T] (already mapped from transition-ids), weights[T] or
 * NULL (=1.0, gmm-acc-stats-ali.cpp:93).  feats2 != NULL selects AccumulateForGmmTwofeats (posteriors from feats,
 * statistics from feats2).  tot_like (nullable) receives this call's sum of weight*loglike. */
int vbgpu_acc_accumulate(vbgpu_acc_t h, const float *feats, const float *feats2, int64_t T, int32_t stride,
                         const int32_t *pdf_ids, const float *weights, double *tot_like);
int vbgpu_acc_accumulate_dev(vbgpu_acc_t h, const float *d_feats, const float *d_feats2, int64_t T, int32_t stride,
                             const int32_t *d_pdf_ids, const float *d_weights, void *stream);
/* The whole accumulator is ONE device buffer of doubles laid out
 *   [ occ (N) | mean_acc (N x D) | var_acc (N x D) | tot_like | tot_frames | transition accs (num_tids + 1, optional) ]
 * so that the per-EM-iteration reduce over GPUs is a single in-place sum all-reduce (replaces gmm-sum-accs.cpp:44-50). */
int vbgpu_acc_buffer(vbgpu_acc_t h, double **d_ptr, int64_t *n_doubles);
/* In-place ncclAllReduce(ncclDouble, ncclSum) of that buffer; comm is an ncclComm_t.  libnccl is resolved at run time
 * (dlopen), so the library itself has no link-time NCCL dependency. */
int vbgpu_acc_allreduce(vbgpu_acc_t h, void *nccl_comm, void *stream);
/* AccumAmDiagGmm::Add(scale, other) (mle-am-diag-gmm.cc:279-287) on the device. */
int vbgpu_acc_add(vbgpu_acc_t h, double scale, vbgpu_acc_t other);
/* Download: occ[N], mean_acc[N*D], var_acc[N*D] (doubles, packed), tot_like, tot_frames. */
int vbgpu_acc_download(vbgpu_acc_t h, double *occ, double *mean_acc, double *var_acc, double *tot_like,
                       double *tot_frames);

/* ---- fMLLR sufficient statistics (SURVEY.md §8f n1) --------------------------------------------------------------------
 * Replaces FmllrDiagGmmAccs::AccumulateForGmm / AccumulateFromPosteriors / CommitSingleFrameStats
 * (transform/fmllr-diag-gmm.cc:30-45,110-121,562-583, update_type "full") as driven per utterance by
 * VB/src/gmmbin/gmm-est-fmllr.cpp:40-55, for all speakers of a batch at once.  The solver
 * (FmllrDiagGmmAccs::Update -> ComputeFmllrMatrixDiagGmmFull) stays on the host and takes these statistics unchanged.
 * One handle holds n_spk independent AffineXformStats (transform/transform-common.h:30-58). */
int vbgpu_fmllr_create(vbgpu_gmm_t model, int32_t n_spk, vbgpu_fmllr_t *out);
int vbgpu_fmllr_destroy(vbgpu_fmllr_t h);
int vbgpu_fmllr_zero(vbgpu_fmllr_t h);
/* AccumulateForGmm(pdf_ids[t], feats row t, weights[t] or 1.0) for every frame; frames [frame_offsets[u],
 * frame_offsets[u+1]) belong to utterance u of speaker utt2spk[u] (NULL = speaker 0).  tot_like (nullable) receives
 * this call's sum of the frames' log-likelihoods (AccumulateForGmm's return values). */
int vbgpu_fmllr_accumulate(vbgpu_fmllr_t h, const float *feats, int64_t T, int32_t stride, const int32_t *pdf_ids,
                           const float *weights, const int64_t *frame_offsets, int32_t n_utts, const int32_t *utt2spk,
                           double *tot_like);
/* Same with device-resident features / pdf ids / weights (frame_offsets and utt2spk stay host arrays). */
int vbgpu_fmllr_accumulate_dev(vbgpu_fmllr_t h, const float *d_feats, int64_t T, int32_t stride,
                               const int32_t *d_pdf_ids, const float *d_weights, const int64_t *frame_offsets,
                               int32_t n_utts, const int32_t *utt2spk, void *stream);
/* One speaker's statistics: beta, K[D x (D+1)] row-major, G[D][(D+1)(D+2)/2] with each G[i] in SpMatrix packing (row-major
 * lower triangle, matrix/packed-matrix.h).  Any output may be NULL. */
int vbgpu_fmllr_download(vbgpu_fmllr_t h, int32_t spk, double *beta, double *K, double *G);
/* MlltAccs::AccumulateFromGmm for every frame of an alignment (transform/mllt.cc:131-170; driver
 * VB/src/gmmbin/gmm-acc-mllt.cpp:100-112), rand_prune = 0 (the reference's randomised pruning is a CPU speed-up; exact here).
 * beta and G[D][D(D+1)/2] (each G[j] in SpMatrix packing) are ADDED to; tot_like (nullable) += sum of weight*loglike.
 * Runs the fMLLR G contraction over one pseudo-frame per (frame, Gaussian of its pdf). */
int vbgpu_mllt_accumulate(vbgpu_gmm_t model, const float *feats, int64_t T, int32_t stride, const int32_t *pdf_ids,
                          const float *weights, double *beta, double *G, double *tot_like);

/* ---- LDA class statistics (acc-lda) ----------------------------------------------------------------------------------
 * LdaEstimate::Accumulate (transform/lda-estimate.cc) for every frame of a batch, one (class, weight) per frame: what
 * ali-to-post | weight-silence-post 0.0 hands acc-lda.  For each frame with weight w != 0 and class c:
 *   zero[c] += w,  first[c][:] += w x,  second += w x x^T (lower triangle, SpMatrix packing: (i, j), i >= j, at i(i+1)/2 + j)
 * all in FP64 with x widened from float first.  Frames of weight exactly 0 are skipped (non-finite features there do no
 * harm); any other weight, negative included, is used as given.  A class id outside [0, C) adds nothing for its frame and
 * is counted.  rand_prune is not emulated: every frame is accumulated exactly.  dim 1 ... 256, num_classes >= 1.
 * The solver (LdaEstimate::Estimate, est-lda) stays on the host and takes these statistics unchanged. */
int vbgpu_lda_create(int32_t num_classes, int32_t dim, int device, vbgpu_lda_t *out); /* LdaEstimate::Init */
int vbgpu_lda_destroy(vbgpu_lda_t h);
int vbgpu_lda_zero(vbgpu_lda_t h); /* ZeroAccumulators */
/* Host form, synchronous: feats [T x stride], class_ids[T], weights[T] or NULL (= 1.0).  Returns VBGPU_ERR_NUMERIC after
 * adding every valid frame when some class id was out of range. */
int vbgpu_lda_accumulate(vbgpu_lda_t h, const float *feats, int64_t T, int32_t stride, const int32_t *class_ids,
                         const float *weights);
int vbgpu_lda_accumulate_dev(vbgpu_lda_t h, const float *d_feats, int64_t T, int32_t stride, const int32_t *d_class_ids,
                             const float *d_weights, void *stream);
/* Invalid class ids seen by _dev calls since the last query; resets the count (synchronises the handle's work). */
int vbgpu_lda_bad_count(vbgpu_lda_t h, int64_t *count);
/* zero[C], first[C x D] row-major, second[D(D+1)/2]; any output may be NULL. */
int vbgpu_lda_download(vbgpu_lda_t h, double *zero, double *first, double *second);
/* The statistics are ONE device buffer [ zero (C) | first (C x D) | second (D(D+1)/2) ], so that merging GPUs is a single
 * in-place sum all-reduce (replaces est-lda summing the per-job accumulator files). */
int vbgpu_lda_buffer(vbgpu_lda_t h, double **d_ptr, int64_t *n_doubles);
/* In-place ncclAllReduce(ncclDouble, ncclSum) of that buffer, resolved at run time as for vbgpu_acc_allreduce. */
int vbgpu_lda_allreduce(vbgpu_lda_t h, void *nccl_comm, void *stream);

/* ---- tree statistics (acc-tree-stats) -----------------------------------------------------------------------------------
 * AccumulateTreeStats (hmm/tree-accu.cc) for a packed batch of whole utterances: transition-ids tids[T] (one per feature
 * row) and rows [frame_offsets[u], frame_offsets[u+1]) of utterance u.  Each alignment is split into phones as
 * SplitToPhones does (hmm/hmm-utils.cc; reordered or not as IsReordered finds); an alignment it calls bad (or one holding a
 * transition-id outside [1, num_tids]) adds nothing, its rows are never read, and it is counted.  Every frame of a good
 * utterance adds GaussClusterable::AddStats(row, 1.0) to its key: count += 1, sum_x += x, sum_x2 += x * x, all FP64.
 * The key (EventType) of a frame in phone segment s: (kPdfClass = -1, pdf-class of its transition-id) and (j, phone of
 * segment s - P + j, 0 outside the utterance) for j = 0 ... N-1, or only (P, central phone) when the central phone is
 * one of ci_phones.  No --phone-map, no frame weights.
 * Limits, checked at create: N <= 4, P < N, phones 1 ... 4095, pdf-classes 0 ... 255, dim 1 ... 256.
 * Keys live in a device hash table of max_keys entries; frames whose key finds no room add nothing and are counted.
 * Every accumulate call sorts frames over the whole id range, at a cost that grows with max_keys: size it to the expected
 * key count (vbgpu_tree_num_keys after a first job tells it). */
#define VBGPU_TID_SELF_LOOP 1       /* IsSelfLoop: the transition's destination is its own hmm-state */
#define VBGPU_TID_FINAL 2           /* IsFinal: destination + 1 == the number of states of the phone's topology entry */
#define VBGPU_TID_STATE0_EMITTING 4 /* state 0 of the phone's topology entry has forward_pdf_class != kNoPdf */
/* Per transition-id tables (vbgpu_io_mdl_transitions fills them from a model file): arrays of num_tids + 1, entry 0
 * unused (transition-ids are 1-based).  pdf_class is the state's self_loop_pdf_class for a self-loop, else its
 * forward_pdf_class; trans_state is the 1-based transition state (tuple index). */
typedef struct vbgpu_tid_tables {
  int32_t num_tids;
  const int32_t *phone, *hmm_state, *pdf_class, *trans_state, *flags;
} vbgpu_tid_tables;
typedef struct vbgpu_tree_opts {
  int32_t context_width;     /* N (acc-tree-stats --context-width, default 3) */
  int32_t central_position;  /* P (--central-position, default 1) */
  const int32_t *ci_phones;  /* --ci-phones, sorted ascending; may be NULL when num_ci_phones == 0 */
  int32_t num_ci_phones;
} vbgpu_tree_opts;
int vbgpu_tree_create(const vbgpu_tree_opts *opts, const vbgpu_tid_tables *tables, int32_t dim, int32_t max_keys,
                      int device, vbgpu_tree_t *out);
int vbgpu_tree_destroy(vbgpu_tree_t h);
int vbgpu_tree_zero(vbgpu_tree_t h); /* empties the statistics and the key table */
/* Host form, synchronous: feats [T x stride], tids[T], T = frame_offsets[n_utts].  Returns VBGPU_ERR_NUMERIC after adding
 * everything else when some frame of this call found no room in the key table. */
int vbgpu_tree_accumulate(vbgpu_tree_t h, const float *feats, int32_t stride, const int32_t *tids,
                          const int64_t *frame_offsets, int32_t n_utts);
/* Device form: d_feats and d_tids on the device, frame_offsets on the host (the batch layout is cached). */
int vbgpu_tree_accumulate_dev(vbgpu_tree_t h, const float *d_feats, int32_t stride, const int32_t *d_tids,
                              const int64_t *frame_offsets, int32_t n_utts, void *stream);
/* Bad utterances (dropped as "alignment appears to be bad") and frames without room in the key table, over every
 * accumulate call since the last query; resets both (synchronises the handle's work).  Either output may be NULL. */
int vbgpu_tree_bad_count(vbgpu_tree_t h, int64_t *bad_utterances, int64_t *dropped_frames);
int vbgpu_tree_num_keys(vbgpu_tree_t h, int32_t *num_keys);
/* The K = num_keys statistics in the order std::map<EventType, GaussClusterable*> iterates them (what acc-tree-stats
 * writes): pdf_class[K], phones[K x N] (-1 where the EventType has no such position), count[K], sum_x[K x D],
 * sum_x2[K x D].  Any output may be NULL. */
int vbgpu_tree_download(vbgpu_tree_t h, int32_t *pdf_class, int32_t *phones, double *count, double *sum_x,
                        double *sum_x2);
/* Adds n entries in the layout of vbgpu_tree_download, key by key (sum-tree-stats; merging the handles of several GPUs,
 * whose keys differ).  Returns VBGPU_ERR_NUMERIC when some entry found no room in the key table. */
int vbgpu_tree_add(vbgpu_tree_t h, int32_t n, const int32_t *pdf_class, const int32_t *phones, const double *count,
                   const double *sum_x, const double *sum_x2);

/* ---- Kaldi wire / disk formats on memory buffers (SURVEY.md §8f n2) ----------------------------------------------------
 * Binary forms only (what the recipes' temp files and archives hold).  Every object may carry the "\0B" marker of
 * WriteKaldiObject / the table holders in front. */
typedef struct vbgpu_io_info {
  int32_t kind;            /* 1 "FM", 2 "DM", 3 "CM" (1 byte + per-column header), 4 "CM2" (2 byte), 5 "CM3" (1 byte),
                              6 "FV", 7 "DV", 8 int32 vector */
  int32_t rows, cols;      /* vectors: rows = 1 */
  float min_value, range;  /* CompressedMatrix::GlobalHeader */
  int64_t header_bytes;    /* offset of the payload from the start of the object (marker included) */
  int64_t total_bytes;     /* size of the whole object */
} vbgpu_io_info;
int vbgpu_io_object_info(const void *buf, int64_t n, vbgpu_io_info *info);
/* Matrix<BaseFloat>::Read / CompressedMatrix::CopyToMat (kaldi-matrix.cc:1375-1460, compressed-matrix.cc:617-670). */
int vbgpu_io_read_matrix(const void *buf, int64_t n, float *out, int32_t out_stride);
int vbgpu_io_read_vector(const void *buf, int64_t n, double *out);
/* BasicVectorHolder<int32> objects (alignments, util/kaldi-holder-inl.h:230-243); returns the element count. */
int vbgpu_io_read_int32_vector(const void *buf, int64_t n, int32_t *out, int32_t cap);
/* Writers return the number of bytes the object takes; nothing is written beyond cap (call with cap = 0 to size). */
int64_t vbgpu_io_write_matrix(const float *data, int32_t rows, int32_t cols, int32_t stride, void *buf, int64_t cap);
int64_t vbgpu_io_write_int32_vector(const int32_t *data, int32_t count, void *buf, int64_t cap);
/* One entry "key \0B<object>" of a binary archive starting at byte pos: 0 = ok, 1 = end of archive. */
int vbgpu_io_ark_next(const void *buf, int64_t n, int64_t pos, char *key, int32_t key_cap, int64_t *obj_pos,
                      int64_t *next_pos, vbgpu_io_info *info);
/* Model file (TransitionModel + AmDiagGmm, hmm/transition-model.cc:383-409, gmm/am-diag-gmm.cc:147-161) or a bare
 * AmDiagGmm.  num_tids = 0 when there is no transition model.  _read fills the flattened model vbgpu_gmm_create takes
 * (gconsts recomputed like DiagGmm::ComputeGconsts, diag-gmm.cc:114-152; returns the number of infinite gconsts) and
 * tid2pdf[num_tids + 1] (entry 0 unused: transition-ids are 1-based).  Any output may be NULL. */
int vbgpu_io_mdl_info(const void *buf, int64_t n, int32_t *dim, int32_t *num_pdfs, int32_t *num_gauss, int32_t *num_tids);
int vbgpu_io_mdl_read(const void *buf, int64_t n, int32_t *pdf_offsets, float *gconsts, float *weights,
                      float *means_invvars, float *inv_vars, int32_t *tid2pdf, float *trans_log_probs);
/* The per transition-id tables of the model file's TransitionModel (the arrays of vbgpu_tid_tables, num_tids + 1 each,
 * entry 0 unused), from its topology (forward / self-loop pdf classes, transitions) and <Triples> or <Tuples>.  Returns
 * num_tids; any output may be NULL. */
int vbgpu_io_mdl_transitions(const void *buf, int64_t n, int32_t *phone, int32_t *hmm_state, int32_t *pdf_class,
                             int32_t *trans_state, int32_t *flags);
/* A statistics file as gmm-acc-stats-ali writes it (gmm-acc-stats-ali.cpp:124-128): transition accs (n_trans may be 0)
 * + AccumAmDiagGmm::Write with flags kGmmAll, doubles narrowed to float (mle-diag-gmm.cc:86-101). */
int64_t vbgpu_io_write_acc(int32_t num_pdfs, int32_t dim, const int32_t *pdf_offsets, const double *trans_accs,
                           int32_t n_trans, const double *occ, const double *mean_acc, const double *var_acc,
                           double tot_like, double tot_frames, void *buf, int64_t cap);
/* A feature matrix object (host bytes, any matrix kind) expanded into a device float matrix: "FM" is one strided copy; the
 * packed kinds cross PCIe as stored (1 or 2 bytes per element) into d_scratch (>= total_bytes - header_bytes) and are
 * expanded by a kernel, bit-identical to CompressedMatrix::CopyToMat. */
int vbgpu_io_matrix_to_device(const void *buf, int64_t n, float *d_out, int32_t out_stride, void *d_scratch,
                              int64_t scratch_bytes, void *stream);

/* ---- fused pipeline: PCM -> log-likelihoods / statistics ---------------------------------------------------------- */
/* Combines one MFCC computer, one feature pipeline and one model (all on the same device; the pipeline borrows them). */
int vbgpu_pipeline_create(vbgpu_mfcc_t mfcc, vbgpu_feat_t feat, vbgpu_gmm_t gmm, vbgpu_pipeline_t *out);
int vbgpu_pipeline_destroy(vbgpu_pipeline_t h);
/* Host form (what a decode job calls): PCM of a batch of whole speakers in, [total_frames x ll_stride] loglikes out.
 * CMVN statistics are computed per speaker from the batch itself unless cmvn_stats != NULL.  Copies and kernels are
 * pipelined in chunks of utterances on two streams through pinned staging buffers.
 * feats_out (nullable): the processed features [total_frames x feats_stride]. */
int vbgpu_pipeline_score_i16(vbgpu_pipeline_t h, const int16_t *pcm, const int64_t *sample_offsets, int32_t n_utts,
                             const int32_t *utt2spk, int32_t n_spk, const double *cmvn_stats, const float *fmllr,
                             int32_t fmllr_cols, float *loglikes, int32_t ll_stride, float *feats_out,
                             int32_t feats_stride);
/* Device form: everything resident; d_loglikes [total_frames x ll_stride]; d_feats (nullable) receives the features. */
int vbgpu_pipeline_score_dev(vbgpu_pipeline_t h, const int16_t *d_pcm, const int64_t *sample_offsets, int32_t n_utts,
                             const int32_t *utt2spk, int32_t n_spk, const float *d_fmllr, int32_t fmllr_cols,
                             float *d_loglikes, int32_t ll_stride, float *d_feats, int32_t feats_stride, void *stream);
/* Same, d_loglikes in device column order (ll_stride >= vbgpu_gmm_num_cols(), see vbgpu_gmm_score_cols_dev). */
int vbgpu_pipeline_score_cols_dev(vbgpu_pipeline_t h, const int16_t *d_pcm, const int64_t *sample_offsets, int32_t n_utts,
                                  const int32_t *utt2spk, int32_t n_spk, const float *d_fmllr, int32_t fmllr_cols,
                                  float *d_loglikes, int32_t ll_stride, float *d_feats, int32_t feats_stride,
                                  void *stream);
/* Host forms for the sparse consumers (see vbgpu_gmm_score_subset / _gather): PCM of a batch in, only the requested
 * log-likelihoods out — what an alignment or rescoring job needs from the path, a few per cent of the dense matrix. */
int vbgpu_pipeline_score_subset_i16(vbgpu_pipeline_t h, const int16_t *pcm, const int64_t *sample_offsets, int32_t n_utts,
                                    const int32_t *utt2spk, int32_t n_spk, const double *cmvn_stats, const float *fmllr,
                                    int32_t fmllr_cols, const int64_t *subset_offsets, const int32_t *subset_pdfs, float *out,
                                    int64_t *out_offsets);
int vbgpu_pipeline_score_gather_i16(vbgpu_pipeline_t h, const int16_t *pcm, const int64_t *sample_offsets, int32_t n_utts,
                                    const int32_t *utt2spk, int32_t n_spk, const double *cmvn_stats, const float *fmllr,
                                    int32_t fmllr_cols, const int32_t *frames, const int32_t *pdfs, int64_t n, float *out);
/* Training form: PCM + alignment in, statistics accumulated into `acc` (PCM -> stats path of cfg 5). */
int vbgpu_pipeline_accumulate_dev(vbgpu_pipeline_t h, vbgpu_acc_t acc, const int16_t *d_pcm,
                                  const int64_t *sample_offsets, int32_t n_utts, const int32_t *utt2spk, int32_t n_spk,
                                  const float *d_fmllr, int32_t fmllr_cols, const int32_t *d_pdf_ids, void *stream);

/* ---- Kaldi pitch (SURVEY.md §8f n4; make_mfcc_pitch / compute-kaldi-pitch-feats / process-kaldi-pitch-feats) ------- *
 * Replaces ComputeKaldiPitch (feat/pitch-functions.cc:1291-1325: LinearResample to resample_freq, per-frame NCCF with the
 * energy ballast, ArbitraryResample onto the log-spaced lag grid, Viterbi over the lags with the RecomputeBacktraces
 * energy correction :945-1035) and ProcessPitch (:1581-1595) for a batch of utterances, offline mode only
 * (frames_per_chunk = 0, simulate_first_pass_online = false, nccf_ballast_online = false, max_frames_latency = 0).
 * Field meanings and defaults are PitchExtractionOptions / ProcessPitchOptions (feat/pitch-functions.h:43-123, 216-255). */
typedef struct vbgpu_pitch_opts {
  float samp_freq;               /* 16000 */
  float frame_shift_ms;          /* 10 */
  float frame_length_ms;         /* 25 */
  float preemph_coeff;           /* 0 */
  float min_f0;                  /* 50 */
  float max_f0;                  /* 400 */
  float soft_min_f0;             /* 10 */
  float penalty_factor;          /* 0.1 */
  float lowpass_cutoff;          /* 1000 */
  float resample_freq;           /* 4000 */
  float delta_pitch;             /* 0.005 */
  float nccf_ballast;            /* 7000 */
  int32_t lowpass_filter_width;  /* 1 */
  int32_t upsample_filter_width; /* 5 */
  int32_t recompute_frame;       /* 500 */
  int32_t snip_edges;            /* 1 */
} vbgpu_pitch_opts;

typedef struct vbgpu_process_pitch_opts {
  float pitch_scale;                   /* 2 */
  float pov_scale;                     /* 2 */
  float pov_offset;                    /* 0 */
  float delta_pitch_scale;             /* 10 */
  float delta_pitch_noise_stddev;      /* 0.005; drawn from a counter-based generator, NOT the reference's rand() stream:
                                          set 0 for results comparable with the reference sample by sample */
  int32_t normalization_left_context;  /* 75 */
  int32_t normalization_right_context; /* 75 */
  int32_t delta_window;                /* 2 */
  int32_t delay;                       /* 0 */
  int32_t add_pov_feature;             /* 1 */
  int32_t add_normalized_log_pitch;    /* 1 */
  int32_t add_delta_pitch;             /* 1 */
  int32_t add_raw_log_pitch;           /* 0 */
} vbgpu_process_pitch_opts;

void vbgpu_pitch_opts_default(vbgpu_pitch_opts *opts);
void vbgpu_process_pitch_opts_default(vbgpu_process_pitch_opts *opts);
int vbgpu_pitch_create(const vbgpu_pitch_opts *opts, int device, vbgpu_pitch_t *out);
void vbgpu_pitch_destroy(vbgpu_pitch_t h);
int32_t vbgpu_pitch_num_states(vbgpu_pitch_t h);                    /* lags searched, SelectLags :157-167 */
int64_t vbgpu_pitch_num_frames(vbgpu_pitch_t h, int64_t n_samples); /* rows ComputeKaldiPitch returns */
/* Batch of n_utts utterances packed in `wave` (sample_offsets[n_utts+1], [0] = 0); wave / out may be host (pageable or
 * pinned) or device memory, sample_offsets is host memory.  process == NULL:
 * out rows are (NCCF at the chosen lag, pitch in Hz), vbgpu_pitch_num_frames() rows per utterance, packed in order.
 * process != NULL: ComputeAndProcessKaldiPitch (:1597-1665) output instead, num_frames + delay rows per non-empty
 * utterance and one column per add_* flag.  out_stride in floats. */
int vbgpu_pitch_compute_f32(vbgpu_pitch_t h, const float *wave, const int64_t *sample_offsets, int32_t n_utts,
                            const vbgpu_process_pitch_opts *process, float *out, int32_t out_stride);
int vbgpu_pitch_compute_i16(vbgpu_pitch_t h, const int16_t *pcm, const int64_t *sample_offsets, int32_t n_utts,
                            const vbgpu_process_pitch_opts *process, float *out, int32_t out_stride);
/* ProcessPitch on (NCCF, pitch) rows supplied by the caller (process-kaldi-pitch-feats). */
int vbgpu_pitch_process(vbgpu_pitch_t h, const vbgpu_process_pitch_opts *process, const float *raw, int32_t raw_stride,
                        const int64_t *frame_offsets, int32_t n_utts, float *out, int32_t out_stride);

#ifdef __cplusplus
}
#endif
#endif /* VBGPU_H_ */
