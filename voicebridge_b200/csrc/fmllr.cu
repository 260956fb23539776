// fmllr.cu — fMLLR sufficient statistics for many speakers at once: FmllrDiagGmmAccs::AccumulateForGmm
// (transform/fmllr-diag-gmm.cc:110-121) -> AccumulateFromPosteriors (:30-45) -> CommitSingleFrameStats (:562-583,
// update_type "full"), driven per utterance by gmm-est-fmllr.cpp:40-55 (one (pdf, weight) per frame after ali-to-post).
// Per frame t of speaker s, with gamma = softmax(loglikes of the aligned pdf) * weight:
//     a_t = sum_g gamma_g means_invvars_g        b_t = sum_g gamma_g inv_vars_g            (FP32, as the reference's sgemv)
//     beta_s += sum_g gamma_g     K_s += a_t (x) [x_t; 1]     G_s[i] += b_t[i] * [x_t; 1][x_t; 1]^T           (FP64)
// SURVEY.md §8f n1.  The solver (ComputeFmllrMatrixDiagGmmFull) stays on the host and consumes these unchanged.
//
// Three kernels:
//   a_t, b_t, count  frames counting-sorted by pdf, then the EM path's bucketed kernel (accum.cu, posterior mode): a CTA per (pdf,
//                    chunk of 128 frames) with the pdf's model rows staged in shared memory; pdfs with more than 64 Gaussians take
//                    fmllr_ab_kernel (warp = frame).
//   fmllr_g_kernel   the heavy part, G[i][j][k] = sum_t b_ti xi_tj xi_tk: a [D x T].[T x npairs] contraction whose second
//                    operand Z_t[(j,k)] = xi_tj xi_tk is formed on the fly in REGISTERS.  CTA = (speaker, chunk of <= 1024
//                    frames, half of the thread tiles); thread tile 8 (i) x one 4 x 2 block of pairs, two CTAs per SM, one
//                    FP64 red.global.add per accumulator per
//                    chunk.  FP32 over <= 1024 terms then FP64 keeps the statistics within ~2e-6 relative of the
//                    reference's all-FP64 sums (budget 1e-4).
//   fmllr_k_kernel   K and beta in FP64 directly (D(D+1) outputs, negligible).
#include <algorithm>
#include <cuda_pipeline.h>

#include <cfloat>
#include <cstdlib>

#include "common.h"

struct vbgpu_fmllr_s {
  vb::StreamOrder order;  // cross-stream ordering of the handle's scratch
  vbgpu_gmm_t model = nullptr;
  int device = 0;
  vb::Stream stream;
  int32_t n_spk = 0, D = 0, np = 0;
  int64_t per_spk = 0;  // doubles per speaker: beta | K[D][D+1] | G[D][np]
  vb::DevBuf d_stats, d_ab, d_cnt, d_units, d_pairs, d_like, d_work;
  vb::DevBuf d_feats, d_ids, d_w;  // staging of the host entry point
  vb::CallCount count;  // the host forms' own errors (the _dev form counts into the model's running count)
  std::vector<int32_t> h_units;
};

namespace {

constexpr int kWarps = 8;
constexpr int kMaxD = 40;       // feature dimension served (39 = delta, 40 = LDA+MLLT)
constexpr int kXi = 48;         // padded [x; 1]
constexpr int kFChunk = 1024;   // frames per work unit: FP32 partial sums over <= 1024 terms (~2e-6 relative), then FP64
constexpr int kFT = 32;         // frames per shared-memory tile of the G kernel
// G kernel: (D+1 = 40) 110 blocks of 4 x 2 pairs x 5 row groups = 550 thread tiles -> 2 CTAs of 288 threads; D + 1 = 41: 660 -> 2 x 352

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sumf(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- per-frame a, b, count ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kWarps * 32) fmllr_ab_kernel(
    const float *__restrict__ feats, int64_t T, int32_t stride, int32_t D, int32_t DP,
    const int32_t *__restrict__ pdf_ids, const float *__restrict__ weights, const float *__restrict__ rows,
    const float *__restrict__ gconsts, const int32_t *__restrict__ pdf_offsets, int32_t P,
    float *__restrict__ ab,   // [T][2*kMaxD]: a | b
    float *__restrict__ cnt,  // [T]
    double *__restrict__ tot_like, unsigned long long *bad, int32_t min_gauss) {
  // min_gauss > 0: only frames whose pdf has more than min_gauss Gaussians (the bucketed kernel of accum.cu served the rest,
  // invalid pdf ids included)
  __shared__ float s_x[kWarps][2 * kMaxD];
  __shared__ float s_post[kWarps][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double like = 0.0;
  unsigned long long nbad = 0;
  for (int64_t t = (int64_t)blockIdx.x * kWarps + warp; t < T; t += (int64_t)gridDim.x * kWarps) {
    float *abr = ab + t * (2 * kMaxD);
    const int p = pdf_ids[t];
    bool ok = p >= 0 && p < P;
    if (min_gauss > 0 && (!ok || pdf_offsets[p + 1] - pdf_offsets[p] <= min_gauss)) continue;
    float log_like = 0.0f, run_max = -INFINITY, run_sum = 0.0f;
    int g0 = 0, M = 0;
    if (ok) {
      const float *xr = feats + t * stride;
      for (int d = lane; d < D; d += 32) {
        const float v = xr[d];
        s_x[warp][d] = v;
        s_x[warp][kMaxD + d] = v * v;
      }
      __syncwarp();
      g0 = pdf_offsets[p], M = pdf_offsets[p + 1] - g0;
      for (int c0 = 0; c0 < M; c0 += 32) {  // lane = Gaussian; online max / sum across chunks of 32
        const int m = c0 + lane;
        float ll = -INFINITY;
        if (m < M) {
          const float *r = rows + (size_t)(g0 + m) * (2 * DP);
          float a = 0.0f, b = 0.0f;
          for (int d = 0; d < D; d++) a = fmaf(r[d], s_x[warp][d], a);
          for (int d = 0; d < D; d++) b = fmaf(r[DP + d], s_x[warp][kMaxD + d], b);
          ll = (gconsts[g0 + m] + a) + b;
        }
        const float nmax = fmaxf(run_max, warp_max(ll));
        const float e = (m < M && nmax > -INFINITY) ? __expf(ll - nmax) : 0.0f;
        run_sum = (run_max > -INFINITY ? run_sum * __expf(run_max - nmax) : 0.0f) + warp_sumf(e);
        run_max = nmax;
      }
      log_like = run_max + __logf(run_sum);  // ComponentPosteriors returns ApplySoftMax's max + Log(sum)
      ok = fabsf(log_like) <= FLT_MAX;       // diag-gmm.cc:609-610 raises KALDI_ERR otherwise
    }
    if (!ok) {  // invalid pdf id or non-finite likelihood: counted as an error, the frame adds nothing
      if (lane == 0) nbad++, cnt[t] = 0.0f;
      for (int d = lane; d < 2 * kMaxD; d += 32) abr[d] = 0.0f;
      __syncwarp();
      continue;
    }
    const float w = weights ? weights[t] : 1.0f, inv_sum = 1.0f / run_sum;
    float a0 = 0.0f, a1 = 0.0f, b0 = 0.0f, b1 = 0.0f, count = 0.0f;  // lane owns dims lane and lane + 32
    for (int c0 = 0; c0 < M; c0 += 32) {
      const int m = c0 + lane;
      float post = 0.0f;
      if (m < M) {
        const float *r = rows + (size_t)(g0 + m) * (2 * DP);
        float a = 0.0f, b = 0.0f;
        for (int d = 0; d < D; d++) a = fmaf(r[d], s_x[warp][d], a);
        for (int d = 0; d < D; d++) b = fmaf(r[DP + d], s_x[warp][kMaxD + d], b);
        post = __expf(((gconsts[g0 + m] + a) + b) - run_max) * inv_sum * w;  // softmax, then posterior.Scale(weight)
      }
      count += warp_sumf(post);  // stats.count += posterior.Sum()
      s_post[warp][lane] = post;
      __syncwarp();
      const int mc = min(32, M - c0);
      for (int k = 0; k < mc; k++) {  // a += means_invvars^T post, b += inv_vars^T post (rows hold -0.5 inv_vars)
        const float g = s_post[warp][k];
        const float *r = rows + (size_t)(g0 + c0 + k) * (2 * DP);
        if (lane < D) a0 = fmaf(g, r[lane], a0), b0 = fmaf(g, -2.0f * r[DP + lane], b0);
        if (lane + 32 < D) a1 = fmaf(g, r[lane + 32], a1), b1 = fmaf(g, -2.0f * r[DP + lane + 32], b1);
      }
      __syncwarp();
    }
    abr[lane] = lane < D ? a0 : 0.0f;
    abr[kMaxD + lane] = lane < D ? b0 : 0.0f;
    if (lane + 32 < kMaxD) {
      abr[lane + 32] = lane + 32 < D ? a1 : 0.0f;
      abr[kMaxD + lane + 32] = lane + 32 < D ? b1 : 0.0f;
    }
    if (lane == 0) cnt[t] = count, like += (double)log_like;
    __syncwarp();
  }
  if (lane == 0 && like != 0.0) atomicAdd(tot_like, like);
  if (nbad) atomicAdd(bad, nbad);
}

// ---- MLLT statistics (gmm-acc-mllt): one row per (frame, Gaussian of its pdf) --------------------------------------------
// MlltAccs::AccumulateFromPosteriors (transform/mllt.cc:131-160): G[j] += (inv_var_gj * gamma_g) (mu_g - x)(mu_g - x)^T.  That is
// the fMLLR G contraction over pseudo-frames: row (t, g) carries xi = mu_g - x_t (FP32, as the reference forms it) and
// b = inv_var_g * gamma_g; fmllr_g_kernel then sums b[j] xi xi^T over the rows.  warp = frame.
template <bool ROWS>  // false: Gaussian-level posteriors only (gmm-post-to-gpost)
__global__ void __launch_bounds__(kWarps * 32) mllt_rows_kernel(
    const float *__restrict__ feats, int64_t T, int32_t stride, int32_t D, int32_t DP, const int32_t *__restrict__ pdf_ids,
    const float *__restrict__ weights, const float *__restrict__ rows, const float *__restrict__ gconsts,
    const int32_t *__restrict__ pdf_offsets, int32_t P, const int32_t *__restrict__ row_off,  // [T + 1]
    float *__restrict__ xi_rows,  // [R][kMaxD]
    float *__restrict__ ab_rows,  // [R][2*kMaxD]: (unused) | b
    float *__restrict__ cnt_rows, double *__restrict__ tot_like, unsigned long long *bad,
    float *__restrict__ frame_like) {  // [T] nullable: ComponentPosteriors' return value per frame
  __shared__ float s_x[kWarps][2 * kMaxD];
  __shared__ float s_post[kWarps][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double like = 0.0;
  unsigned long long nbad = 0;
  for (int64_t t = (int64_t)blockIdx.x * kWarps + warp; t < T; t += (int64_t)gridDim.x * kWarps) {
    const int p = pdf_ids[t];
    if (p < 0 || p >= P) {
      if (lane == 0) nbad++;
      if (lane == 0 && frame_like) frame_like[t] = 0.0f;
      continue;
    }
    const float *xr = feats + t * stride;
    for (int d = lane; d < D; d += 32) {
      const float v = xr[d];
      s_x[warp][d] = v;
      s_x[warp][kMaxD + d] = v * v;
    }
    __syncwarp();
    const int g0 = pdf_offsets[p], M = pdf_offsets[p + 1] - g0;
    float run_max = -INFINITY, run_sum = 0.0f;
    for (int c0 = 0; c0 < M; c0 += 32) {
      const int m = c0 + lane;
      float ll = -INFINITY;
      if (m < M) {
        const float *r = rows + (size_t)(g0 + m) * (2 * DP);
        float a = 0.0f, b = 0.0f;
        for (int d = 0; d < D; d++) a = fmaf(r[d], s_x[warp][d], a);
        for (int d = 0; d < D; d++) b = fmaf(r[DP + d], s_x[warp][kMaxD + d], b);
        ll = (gconsts[g0 + m] + a) + b;
      }
      const float nmax = fmaxf(run_max, warp_max(ll));
      const float e = (m < M && nmax > -INFINITY) ? __expf(ll - nmax) : 0.0f;
      run_sum = (run_max > -INFINITY ? run_sum * __expf(run_max - nmax) : 0.0f) + warp_sumf(e);
      run_max = nmax;
    }
    const float log_like = run_max + __logf(run_sum);
    const int64_t row0 = row_off[t];
    if (lane == 0 && frame_like) frame_like[t] = log_like;
    if (!(fabsf(log_like) <= FLT_MAX)) {  // ComponentPosteriors raises KALDI_ERR: reported, the frame's rows stay zero
      if (lane == 0) nbad++;
      __syncwarp();
      continue;
    }
    const float w = weights ? weights[t] : 1.0f, inv_sum = 1.0f / run_sum;
    for (int c0 = 0; c0 < M; c0 += 32) {
      const int m = c0 + lane;
      float post = 0.0f;
      if (m < M) {
        const float *r = rows + (size_t)(g0 + m) * (2 * DP);
        float a = 0.0f, b = 0.0f;
        for (int d = 0; d < D; d++) a = fmaf(r[d], s_x[warp][d], a);
        for (int d = 0; d < D; d++) b = fmaf(r[DP + d], s_x[warp][kMaxD + d], b);
        post = __expf(((gconsts[g0 + m] + a) + b) - run_max) * inv_sum * w;
        cnt_rows[row0 + m] = post;
      }
      if (!ROWS) continue;
      s_post[warp][lane] = post;
      __syncwarp();
      const int mc = min(32, M - c0);
      for (int k = 0; k < mc; k++) {
        const float g = s_post[warp][k];
        const float *r = rows + (size_t)(g0 + c0 + k) * (2 * DP);
        const int64_t row = row0 + c0 + k;
        for (int d = lane; d < D; d += 32) {
          const float iv = -2.0f * r[DP + d];                         // the rows hold -0.5 inv_vars
          const float mean = __fdiv_rn(r[d], iv);                     // mean.AddVecDivVec(1.0, mean_invvar, inv_var, 0.0)
          xi_rows[row * kMaxD + d] = __fadd_rn(mean, -s_x[warp][d]);  // mean.AddVec(-1.0, data)
          ab_rows[row * (2 * kMaxD) + kMaxD + d] = __fmul_rn(iv, g);  // inv_var(j) * posterior
        }
      }
      __syncwarp();
    }
    if (lane == 0) like += (double)(log_like * w);
    __syncwarp();
  }
  if (lane == 0 && like != 0.0) atomicAdd(tot_like, like);
  if (nbad) atomicAdd(bad, nbad);
}

// ---- G: grid (unit, half of the thread tiles) --------------------------------------------------------------------------
// The (D+1) x (D+1) symmetric matrix of pair products is cut into blocks of 4 (j) x 2 (k); a thread owns one block of the
// lower triangle and 8 output rows i, i.e. acc[i][a][c] = sum_t b_t[i] xi_t[4jb+a] xi_t[2kb+c].  Per frame it reads xi of its
// block row (float4), of its block column (float2) and 8 b's from shared memory, forms the 8 products in registers and issues
// 64 FMAs.  64 accumulators keep the kernel under 112 registers, so two CTAs (each with half of the thread tiles) share an
// SM, and each stages its next 32 frames with cp.async into a second buffer while it computes on the first.
template <int THREADS>
__global__ void __launch_bounds__(THREADS, 2) fmllr_g_kernel(const float *__restrict__ feats, int32_t stride, int32_t D,
                                                             const float *__restrict__ ab, const int32_t *__restrict__ units,
                                                             int32_t n_blocks, int32_t tiles_per_cta, int32_t np,
                                                             double *__restrict__ stats, int64_t per_spk) {
  __shared__ __align__(16) float s_xi[2][kFT][kXi];   // double-buffered: cp.async fills one tile while the other is consumed
  __shared__ __align__(16) float s_b[2][kFT][kMaxD];
  const int tid = threadIdx.x;
  const int spk = units[3 * blockIdx.x], t0 = units[3 * blockIdx.x + 1], n = units[3 * blockIdx.x + 2];
  const int tile = blockIdx.y * tiles_per_cta + tid;           // thread tile = (row group ig, pair block blk)
  const int ig = tile / n_blocks, blk = tile - ig * n_blocks;
  int jb = 0;                                                   // blk = jb (jb + 1) + kb, 0 <= kb <= 2 jb + 1
  while ((jb + 1) * (jb + 2) <= blk) jb++;
  const int kb = blk - jb * (jb + 1);
  const bool active = tid < tiles_per_cta && ig * 8 < D;        // the rest only help with the staging
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; i++)
#pragma unroll
    for (int p = 0; p < 8; p++) acc[i][p] = 0.0f;

  // Stage frames [f0, f0 + kFT) of the unit into buffer `buf`: real elements by cp.async (no register round trip, so the
  // loads of a whole tile are in flight at once), padding / the constant 1 / frames beyond the unit by plain stores.
  auto stage = [&](int f0, int buf) {
    const int nf = min(kFT, n - f0);
    for (int idx = tid; idx < kFT * kXi; idx += THREADS) {
      const int f = idx / kXi, d = idx - f * kXi;
      if (f < nf && d < D) __pipeline_memcpy_async(&s_xi[buf][f][d], feats + (int64_t)(t0 + f0 + f) * stride + d, 4);
      else s_xi[buf][f][d] = (f < nf && d == D) ? 1.0f : 0.0f;
    }
    for (int idx = tid; idx < kFT * kMaxD; idx += THREADS) {
      const int f = idx / kMaxD, i = idx - f * kMaxD;
      if (f < nf) __pipeline_memcpy_async(&s_b[buf][f][i], ab + (int64_t)(t0 + f0 + f) * (2 * kMaxD) + kMaxD + i, 4);
      else s_b[buf][f][i] = 0.0f;
    }
    __pipeline_commit();
  };
  stage(0, 0);
  int buf = 0;
  for (int f0 = 0; f0 < n; f0 += kFT, buf ^= 1) {
    const bool more = f0 + kFT < n;
    if (more) stage(f0 + kFT, buf ^ 1);  // (its previous contents were consumed before the barrier that ended the last round)
    __pipeline_wait_prior(more ? 1 : 0);
    __syncthreads();
    if (active) {
#pragma unroll 1
      for (int f = 0; f < kFT; f++) {  // frames beyond the unit are zero rows: they add nothing
        const float4 xj = *reinterpret_cast<const float4 *>(&s_xi[buf][f][4 * jb]);
        const float2 xk = *reinterpret_cast<const float2 *>(&s_xi[buf][f][2 * kb]);
        const float4 b0 = *reinterpret_cast<const float4 *>(&s_b[buf][f][ig * 8]);
        const float4 b1 = *reinterpret_cast<const float4 *>(&s_b[buf][f][ig * 8 + 4]);
        const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
        const float z[8] = {xj.x * xk.x, xj.x * xk.y, xj.y * xk.x, xj.y * xk.y, xj.z * xk.x, xj.z * xk.y, xj.w * xk.x, xj.w * xk.y};
#pragma unroll
        for (int i = 0; i < 8; i++)
#pragma unroll
          for (int p = 0; p < 8; p++) acc[i][p] = fmaf(b[i], z[p], acc[i][p]);
      }
    }
    __syncthreads();  // this buffer is free for the tile after next
  }
  if (!active) return;
  double *G = stats + (int64_t)spk * per_spk + 1 + (int64_t)D * (D + 1);
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const int gi = ig * 8 + i;
    if (gi >= D) continue;
#pragma unroll
    for (int p = 0; p < 8; p++) {
      const int j = 4 * jb + (p >> 1), k = 2 * kb + (p & 1);
      if (j <= D && k <= j && acc[i][p] != 0.0f) atomicAdd(&G[(int64_t)gi * np + j * (j + 1) / 2 + k], (double)acc[i][p]);
    }
  }
}

// ---- K and beta: grid (unit) -------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) fmllr_k_kernel(const float *__restrict__ feats, int32_t stride, int32_t D,
                                                      const float *__restrict__ ab, const float *__restrict__ cnt,
                                                      const int32_t *__restrict__ units, double *__restrict__ stats,
                                                      int64_t per_spk) {
  constexpr int kT = 32, kE = 7;  // frames per tile; (i, k) entries per thread: 7 * 256 >= 40 * 41
  __shared__ double s_a[kT][kMaxD], s_xi[kT][kXi];  // widened once per element while staging, not once per product
  __shared__ float s_c[kT];
  const int tid = threadIdx.x;
  const int spk = units[3 * blockIdx.x], t0 = units[3 * blockIdx.x + 1], n = units[3 * blockIdx.x + 2];
  const int ne = D * (D + 1);
  int ei[kE], ek[kE];
  double acc[kE];
#pragma unroll
  for (int r = 0; r < kE; r++) {
    const int e = tid + 256 * r;
    ei[r] = e < ne ? e / (D + 1) : 0;
    ek[r] = e < ne ? e - ei[r] * (D + 1) : 0;
    acc[r] = 0.0;
  }
  double beta = 0.0;
  for (int f0 = 0; f0 < n; f0 += kT) {
    const int nf = min(kT, n - f0);
    __syncthreads();
    float vx[kT * kXi / 256], va[kT * kMaxD / 256];  // all loads of the tile in flight before the first store
#pragma unroll
    for (int it = 0; it < kT * kXi / 256; it++) {
      const int idx = tid + it * 256, f = idx / kXi, d = idx - f * kXi;
      vx[it] = 0.0f;
      if (f < nf) vx[it] = d < D ? feats[(int64_t)(t0 + f0 + f) * stride + d] : (d == D ? 1.0f : 0.0f);
    }
#pragma unroll
    for (int it = 0; it < kT * kMaxD / 256; it++) {
      const int idx = tid + it * 256, f = idx / kMaxD, i = idx - f * kMaxD;
      va[it] = f < nf ? ab[(int64_t)(t0 + f0 + f) * (2 * kMaxD) + i] : 0.0f;
    }
    const float vc = (tid < kT && tid < nf) ? cnt[t0 + f0 + tid] : 0.0f;
#pragma unroll
    for (int it = 0; it < kT * kXi / 256; it++) (&s_xi[0][0])[tid + it * 256] = (double)vx[it];
#pragma unroll
    for (int it = 0; it < kT * kMaxD / 256; it++) (&s_a[0][0])[tid + it * 256] = (double)va[it];
    if (tid < kT) s_c[tid] = vc;
    __syncthreads();
    for (int f = 0; f < nf; f++) {
#pragma unroll
      for (int r = 0; r < kE; r++) acc[r] += s_a[f][ei[r]] * s_xi[f][ek[r]];  // K_.AddVecVec(1.0, a, xplus)
    }
    if (tid == 0)
      for (int f = 0; f < nf; f++) beta += (double)s_c[f];  // beta_ += stats.count
  }
  double *base = stats + (int64_t)spk * per_spk;
#pragma unroll
  for (int r = 0; r < kE; r++) {
    const int e = tid + 256 * r;
    if (e < ne && acc[r] != 0.0) atomicAdd(&base[1 + e], acc[r]);
  }
  if (tid == 0 && beta != 0.0) atomicAdd(&base[0], beta);
}

// G, K and beta of the units in h->d_units over rows `d_rows` (features or MLLT pseudo-frames) with a, b, count in h->d_ab / d_cnt.
int launch_gk(vbgpu_fmllr_t h, const float *d_rows, int32_t stride, int n_units, cudaStream_t s) {
  vbgpu_gmm_t g = h->model;
  const int jb_n = (g->D + 1 + 3) / 4, n_blocks = jb_n * (jb_n + 1), ig_n = (g->D + 7) / 8;
  const int tiles = n_blocks * ig_n, tiles_per_cta = (tiles + 1) / 2;
  if (tiles_per_cta <= 288)
    fmllr_g_kernel<288><<<dim3(n_units, 2), 288, 0, s>>>(d_rows, stride, g->D, h->d_ab.as<float>(), h->d_units.as<int32_t>(),
                                                        n_blocks, tiles_per_cta, h->np, h->d_stats.as<double>(), h->per_spk);
  else
    fmllr_g_kernel<352><<<dim3(n_units, 2), 352, 0, s>>>(d_rows, stride, g->D, h->d_ab.as<float>(), h->d_units.as<int32_t>(),
                                                        n_blocks, tiles_per_cta, h->np, h->d_stats.as<double>(), h->per_spk);
  VB_CUDA(cudaGetLastError());
  fmllr_k_kernel<<<n_units, 256, 0, s>>>(d_rows, stride, g->D, h->d_ab.as<float>(), h->d_cnt.as<float>(),
                                         h->d_units.as<int32_t>(), h->d_stats.as<double>(), h->per_spk);
  VB_CUDA(cudaGetLastError());
  return 0;
}

int launch_all(vbgpu_fmllr_t h, const float *d_feats, int64_t T, int32_t stride, const int32_t *d_ids, const float *d_w,
               const int64_t *frame_offsets, int32_t n_utts, const int32_t *utt2spk, unsigned long long *bad,
               cudaStream_t s) {
  vbgpu_gmm_t g = h->model;
  if (T >= (int64_t)1 << 31) return vb::fail(VBGPU_ERR_INVALID, "more than 2^31 frames in one call");
  // work units: (speaker, first frame, frames <= kFChunk); adjacent utterances of one speaker form one run of frames
  std::vector<int32_t> &u = h->h_units;
  u.clear();
  int64_t run_a = 0, run_b = 0;
  int32_t run_spk = -1;
  auto flush_run = [&]() {
    for (int64_t t = run_a; t < run_b; t += kFChunk) {
      u.push_back(run_spk);
      u.push_back((int32_t)t);
      u.push_back((int32_t)std::min<int64_t>(kFChunk, run_b - t));
    }
  };
  for (int32_t i = 0; i < n_utts; i++) {
    const int64_t a = frame_offsets[i], b = frame_offsets[i + 1];
    const int32_t spk = utt2spk ? utt2spk[i] : 0;
    if (a < 0 || b < a || b > T) return vb::fail(VBGPU_ERR_INVALID, "frame_offsets of utterance %d outside [0, T]", i);
    if (spk < 0 || spk >= h->n_spk) return vb::fail(VBGPU_ERR_INVALID, "utt2spk[%d] = %d outside [0, %d)", i, spk, h->n_spk);
    if (b == a) continue;
    if (spk == run_spk && a == run_b) {
      run_b = b;
    } else {
      flush_run();
      run_spk = spk, run_a = a, run_b = b;
    }
  }
  flush_run();
  const int n_units = (int)(u.size() / 3);
  VB_TRY(h->d_ab.reserve((size_t)T * 2 * kMaxD * 4));
  VB_TRY(h->d_cnt.reserve((size_t)T * 4));
  if (n_units == 0) return 0;
  VB_TRY(h->d_units.reserve(u.size() * 4));
  VB_CUDA(cudaMemcpyAsync(h->d_units.p, u.data(), u.size() * 4, cudaMemcpyHostToDevice, s));
  const int sms = vb::num_sms(h->device);
  // a, b, count: frames sorted by pdf and served (pdf, chunk) at a time by the EM path's bucketed kernel in posterior mode;
  // pdfs too large for it take the frame-at-a-time kernel.  Frames neither touches (invalid pdf ids) stay zero.
  VB_CUDA(cudaMemsetAsync(h->d_ab.p, 0, (size_t)T * 2 * kMaxD * 4, s));
  VB_CUDA(cudaMemsetAsync(h->d_cnt.p, 0, (size_t)T * 4, s));
  int32_t served = 0;
  const bool framewise = getenv("VBGPU_ACC_FRAMEWISE") != nullptr;
  if (!framewise)
    VB_TRY(vb::acc_posterior_ab_launch(g, &h->d_work, d_feats, T, stride, d_ids, d_w, h->d_ab.as<float>(), kMaxD,
                                       h->d_cnt.as<float>(), h->d_like.as<double>(), &served, bad, s));
  if (framewise || g->max_pdf_size > served) {
    const int grid = (int)std::min<int64_t>((T + kWarps - 1) / kWarps, (int64_t)sms * 8);
    fmllr_ab_kernel<<<grid, kWarps * 32, 0, s>>>(d_feats, T, stride, g->D, g->DP, d_ids, d_w, g->d_rows.as<float>(),
                                                 g->d_gconsts.as<float>(), g->d_pdf_offsets.as<int32_t>(), g->P,
                                                 h->d_ab.as<float>(), h->d_cnt.as<float>(), h->d_like.as<double>(), bad,
                                                 served);
    VB_CUDA(cudaGetLastError());
  }
  VB_TRY(launch_gk(h, d_feats, stride, n_units, s));
  // (h_units is pageable: cudaMemcpyAsync has staged it before returning, so the next call may overwrite it)
  return 0;
}

}  // namespace

using vb::DeviceGuard;
using vb::fail;

extern "C" {

int vbgpu_fmllr_create(vbgpu_gmm_t model, int32_t n_spk, vbgpu_fmllr_t *out) {
  VB_CHECK(model && out && n_spk >= 1, "bad argument");
  *out = nullptr;
  VB_CHECK(model->D <= kMaxD, "fMLLR statistics serve feature dims up to %d (got %d)", kMaxD, model->D);
  DeviceGuard g(model->device);
  std::unique_ptr<vbgpu_fmllr_s, decltype(&vbgpu_fmllr_destroy)> h(new vbgpu_fmllr_s, vbgpu_fmllr_destroy);
  h->model = model;
  h->device = model->device;
  h->n_spk = n_spk;
  h->D = model->D;
  h->np = (h->D + 1) * (h->D + 2) / 2;
  h->per_spk = 1 + (int64_t)h->D * (h->D + 1) + (int64_t)h->D * h->np;
  std::vector<uint8_t> pairs((size_t)2 * h->np);
  for (int j = 0; j <= h->D; j++)  // SpMatrix packing: (j, k), k <= j, at j(j+1)/2 + k
    for (int k = 0; k <= j; k++) pairs[2 * (j * (j + 1) / 2 + k)] = (uint8_t)j, pairs[2 * (j * (j + 1) / 2 + k) + 1] = (uint8_t)k;
  VB_TRY(h->stream.create());
  const size_t bytes = (size_t)n_spk * h->per_spk * 8;
  VB_TRY(h->d_stats.reserve(bytes));
  VB_TRY(h->d_pairs.upload(pairs.data(), pairs.size()));
  VB_TRY(h->d_like.reserve(8));
  VB_CUDA(cudaMemset(h->d_stats.p, 0, bytes));
  VB_CUDA(cudaMemset(h->d_like.p, 0, 8));
  *out = h.release();
  return 0;
}

int vbgpu_fmllr_destroy(vbgpu_fmllr_t h) {
  if (!h) return 0;
  DeviceGuard g(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  delete h;
  return 0;
}

int vbgpu_fmllr_zero(vbgpu_fmllr_t h) {
  VB_CHECK(h, "null handle");
  DeviceGuard g(h->device);
  VB_CUDA(cudaDeviceSynchronize());
  VB_CUDA(cudaMemset(h->d_stats.p, 0, (size_t)h->n_spk * h->per_spk * 8));
  VB_CUDA(cudaMemset(h->d_like.p, 0, 8));
  return 0;
}

int vbgpu_fmllr_accumulate_dev(vbgpu_fmllr_t h, const float *d_feats, int64_t T, int32_t stride, const int32_t *d_pdf_ids,
                               const float *d_weights, const int64_t *frame_offsets, int32_t n_utts,
                               const int32_t *utt2spk, void *stream) {
  VB_CHECK(h && T >= 0 && n_utts >= 0, "bad argument");
  VB_CHECK(stride >= h->D, "stride %d < D %d", stride, h->D);
  if (T == 0 || n_utts == 0) return 0;
  VB_CHECK(d_feats && d_pdf_ids && frame_offsets, "null buffer");
  DeviceGuard g(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  VB_TRY(h->order.enter(s));
  VB_TRY(launch_all(h, d_feats, T, stride, d_pdf_ids, d_weights, frame_offsets, n_utts, utt2spk,
                    h->model->d_bad.as<unsigned long long>(), s));
  return h->order.leave(s);
}

int vbgpu_fmllr_accumulate(vbgpu_fmllr_t h, const float *feats, int64_t T, int32_t stride, const int32_t *pdf_ids,
                           const float *weights, const int64_t *frame_offsets, int32_t n_utts, const int32_t *utt2spk,
                           double *tot_like) {
  VB_CHECK(h && T >= 0 && n_utts >= 0, "bad argument");
  VB_CHECK(stride >= h->D, "stride %d < D %d", stride, h->D);
  if (tot_like) *tot_like = 0.0;
  if (T == 0 || n_utts == 0) return 0;
  VB_CHECK(feats && pdf_ids && frame_offsets, "null buffer");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  const size_t fb = (size_t)T * stride * 4;
  VB_TRY(h->d_feats.reserve(fb));
  VB_TRY(h->d_ids.reserve((size_t)T * 4));
  VB_CUDA(cudaMemcpyAsync(h->d_feats.p, feats, fb, cudaMemcpyHostToDevice, s));
  VB_CUDA(cudaMemcpyAsync(h->d_ids.p, pdf_ids, (size_t)T * 4, cudaMemcpyHostToDevice, s));
  const float *d_w = nullptr;
  if (weights) {
    VB_TRY(h->d_w.reserve((size_t)T * 4));
    VB_CUDA(cudaMemcpyAsync(h->d_w.p, weights, (size_t)T * 4, cudaMemcpyHostToDevice, s));
    d_w = h->d_w.as<float>();
  }
  double before = 0.0, after = 0.0;
  unsigned long long *bad = nullptr, n_bad = 0;
  VB_CUDA(cudaMemcpyAsync(&before, h->d_like.p, 8, cudaMemcpyDeviceToHost, s));
  VB_TRY(h->count.begin(s, &bad));
  VB_TRY(launch_all(h, h->d_feats.as<float>(), T, stride, h->d_ids.as<int32_t>(), d_w, frame_offsets, n_utts, utt2spk, bad,
                    s));
  VB_CUDA(cudaMemcpyAsync(&after, h->d_like.p, 8, cudaMemcpyDeviceToHost, s));
  VB_TRY(h->count.end(s, &n_bad));
  if (tot_like) *tot_like = after - before;
  if (n_bad) return fail(VBGPU_ERR_NUMERIC, "%llu frames had an invalid pdf-id or a NaN/Inf likelihood", n_bad);
  return 0;
}

int vbgpu_fmllr_download(vbgpu_fmllr_t h, int32_t spk, double *beta, double *K, double *G) {
  VB_CHECK(h && spk >= 0 && spk < h->n_spk, "bad argument");
  DeviceGuard g(h->device);
  VB_CUDA(cudaDeviceSynchronize());
  const double *base = h->d_stats.as<double>() + (int64_t)spk * h->per_spk;
  const size_t nk = (size_t)h->D * (h->D + 1), ng = (size_t)h->D * h->np;
  if (beta) VB_CUDA(cudaMemcpy(beta, base, 8, cudaMemcpyDeviceToHost));
  if (K) VB_CUDA(cudaMemcpy(K, base + 1, nk * 8, cudaMemcpyDeviceToHost));
  if (G) VB_CUDA(cudaMemcpy(G, base + 1 + nk, ng * 8, cudaMemcpyDeviceToHost));
  return 0;
}

int vbgpu_mllt_accumulate(vbgpu_gmm_t model, const float *feats, int64_t T, int32_t stride, const int32_t *pdf_ids,
                          const float *weights, double *beta, double *G, double *tot_like) {
  VB_CHECK(model && T >= 0 && beta && G, "bad argument");
  VB_CHECK(stride >= model->D, "stride %d < D %d", stride, model->D);
  if (T == 0) return 0;
  VB_CHECK(feats && pdf_ids, "null buffer");
  DeviceGuard guard(model->device);
  vbgpu_fmllr_t raw = nullptr;
  VB_TRY(vbgpu_fmllr_create(model, 1, &raw));  // one "speaker": beta | (unused K) | G of the pseudo-frames
  std::unique_ptr<vbgpu_fmllr_s, decltype(&vbgpu_fmllr_destroy)> h(raw, vbgpu_fmllr_destroy);
  cudaStream_t s = h->stream;
  const int D = model->D, P = model->P, sms = vb::num_sms(h->device);
  const std::vector<int32_t> &po = model->h_pdf_offsets;
  vb::DevBuf d_xi, d_off;
  std::vector<int32_t> off;
  unsigned long long *bad = nullptr, n_bad = 0;
  VB_TRY(h->count.begin(s, &bad));
  const int64_t kMaxFrames = 262144, kMaxRows = 1500000;
  for (int64_t t0 = 0; t0 < T;) {
    // a slab of frames whose (frame, Gaussian) rows fit the row buffers
    off.assign(1, 0);
    int64_t t1 = t0;
    while (t1 < T && t1 - t0 < kMaxFrames) {
      const int32_t p = pdf_ids[t1];
      const int32_t M = (p >= 0 && p < P) ? po[p + 1] - po[p] : 0;
      if (off.back() + M > kMaxRows && t1 > t0) break;
      off.push_back(off.back() + M);
      t1++;
    }
    const int64_t n = t1 - t0, R = off.back();
    VB_TRY(h->d_feats.reserve((size_t)n * stride * 4));
    VB_TRY(h->d_ids.reserve((size_t)n * 4));
    VB_TRY(d_off.reserve((size_t)(n + 1) * 4));
    VB_CUDA(cudaMemcpyAsync(h->d_feats.p, feats + t0 * stride, (size_t)n * stride * 4, cudaMemcpyHostToDevice, s));
    VB_CUDA(cudaMemcpyAsync(h->d_ids.p, pdf_ids + t0, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    VB_CUDA(cudaMemcpyAsync(d_off.p, off.data(), (size_t)(n + 1) * 4, cudaMemcpyHostToDevice, s));
    const float *d_w = nullptr;
    if (weights) {
      VB_TRY(h->d_w.reserve((size_t)n * 4));
      VB_CUDA(cudaMemcpyAsync(h->d_w.p, weights + t0, (size_t)n * 4, cudaMemcpyHostToDevice, s));
      d_w = h->d_w.as<float>();
    }
    if (R > 0) {
      VB_TRY(d_xi.reserve((size_t)R * kMaxD * 4));
      VB_TRY(h->d_ab.reserve((size_t)R * 2 * kMaxD * 4));
      VB_TRY(h->d_cnt.reserve((size_t)R * 4));
      VB_CUDA(cudaMemsetAsync(d_xi.p, 0, (size_t)R * kMaxD * 4, s));
      VB_CUDA(cudaMemsetAsync(h->d_ab.p, 0, (size_t)R * 2 * kMaxD * 4, s));
      VB_CUDA(cudaMemsetAsync(h->d_cnt.p, 0, (size_t)R * 4, s));
    }
    const int grid = (int)std::min<int64_t>((n + kWarps - 1) / kWarps, (int64_t)sms * 8);
    mllt_rows_kernel<true><<<grid, kWarps * 32, 0, s>>>(
        h->d_feats.as<float>(), n, stride, D, model->DP, h->d_ids.as<int32_t>(), d_w, model->d_rows.as<float>(),
        model->d_gconsts.as<float>(), model->d_pdf_offsets.as<int32_t>(), P, d_off.as<int32_t>(), d_xi.as<float>(),
        h->d_ab.as<float>(), h->d_cnt.as<float>(), h->d_like.as<double>(), bad, nullptr);
    VB_CUDA(cudaGetLastError());
    if (R > 0) {
      std::vector<int32_t> &u = h->h_units;
      u.clear();
      for (int64_t r0 = 0; r0 < R; r0 += kFChunk) {
        u.push_back(0);
        u.push_back((int32_t)r0);
        u.push_back((int32_t)std::min<int64_t>(kFChunk, R - r0));
      }
      VB_TRY(h->d_units.reserve(u.size() * 4));
      VB_CUDA(cudaMemcpyAsync(h->d_units.p, u.data(), u.size() * 4, cudaMemcpyHostToDevice, s));
      VB_TRY(launch_gk(h.get(), d_xi.as<float>(), kMaxD, (int)(u.size() / 3), s));
    }
    VB_CUDA(cudaStreamSynchronize(s));  // the host staging vectors are rebuilt for the next slab
    t0 = t1;
  }
  // beta | K (ignored) | G[i] packed over (D+1): its first D(D+1)/2 entries are the D x D block MlltAccs keeps
  const int np1 = (D + 1) * (D + 2) / 2, np = D * (D + 1) / 2;
  std::vector<double> st((size_t)h->per_spk);
  double like = 0.0;
  VB_TRY(h->count.end(s, &n_bad));
  VB_CUDA(cudaMemcpy(st.data(), h->d_stats.p, st.size() * 8, cudaMemcpyDeviceToHost));
  VB_CUDA(cudaMemcpy(&like, h->d_like.p, 8, cudaMemcpyDeviceToHost));
  *beta += st[0];
  const double *g = st.data() + 1 + (size_t)D * (D + 1);
  for (int i = 0; i < D; i++)
    for (int k = 0; k < np; k++) G[(size_t)i * np + k] += g[(size_t)i * np1 + k];
  if (tot_like) *tot_like += like;
  if (n_bad) return fail(VBGPU_ERR_NUMERIC, "%llu frames had an invalid pdf-id or a NaN/Inf likelihood", n_bad);
  return 0;
}

int vbgpu_gmm_component_posteriors(vbgpu_gmm_t model, const float *feats, int64_t T, int32_t stride, const int32_t *pdf_ids,
                                   const float *weights, float *post, float *loglikes) {
  VB_CHECK(model && T >= 0, "bad argument");
  VB_CHECK(stride >= model->D && model->D <= kMaxD, "stride %d < D %d, or D > %d", stride, model->D, kMaxD);
  if (T == 0) return 0;
  VB_CHECK(feats && pdf_ids && post, "null buffer");
  VB_CHECK(T < ((int64_t)1 << 31), "more than 2^31 frames in one call");
  DeviceGuard guard(model->device);
  const int P = model->P, sms = vb::num_sms(model->device);
  const std::vector<int32_t> &po = model->h_pdf_offsets;
  std::vector<int32_t> off(1, 0);
  off.reserve((size_t)T + 1);
  for (int64_t t = 0; t < T; t++) {
    const int32_t p = pdf_ids[t];
    const int64_t nx = (int64_t)off.back() + ((p >= 0 && p < P) ? po[p + 1] - po[p] : 0);
    VB_CHECK(nx < ((int64_t)1 << 31), "more than 2^31 posteriors in one call");
    off.push_back((int32_t)nx);
  }
  const int64_t R = off.back();
  vb::DevBuf d_f, d_i, d_w, d_o, d_p, d_l, d_like;
  vb::CallCount count;  // on the legacy default stream, like every copy and the launch below
  unsigned long long *bad = nullptr, n_bad = 0;
  VB_TRY(d_f.reserve((size_t)T * stride * 4));
  VB_TRY(d_i.reserve((size_t)T * 4));
  VB_TRY(d_o.reserve((size_t)(T + 1) * 4));
  VB_TRY(d_p.reserve((size_t)std::max<int64_t>(R, 1) * 4));
  VB_TRY(d_l.reserve((size_t)T * 4));
  VB_TRY(d_like.reserve(8));
  VB_CUDA(cudaMemcpy(d_f.p, feats, (size_t)T * stride * 4, cudaMemcpyHostToDevice));
  VB_CUDA(cudaMemcpy(d_i.p, pdf_ids, (size_t)T * 4, cudaMemcpyHostToDevice));
  VB_CUDA(cudaMemcpy(d_o.p, off.data(), (size_t)(T + 1) * 4, cudaMemcpyHostToDevice));
  VB_CUDA(cudaMemset(d_p.p, 0, (size_t)std::max<int64_t>(R, 1) * 4));
  VB_CUDA(cudaMemset(d_like.p, 0, 8));
  VB_TRY(count.begin(0, &bad));
  const float *dw = nullptr;
  if (weights) {
    VB_TRY(d_w.reserve((size_t)T * 4));
    VB_CUDA(cudaMemcpy(d_w.p, weights, (size_t)T * 4, cudaMemcpyHostToDevice));
    dw = d_w.as<float>();
  }
  const int grid = (int)std::min<int64_t>((T + kWarps - 1) / kWarps, (int64_t)sms * 8);
  mllt_rows_kernel<false><<<grid, kWarps * 32>>>(d_f.as<float>(), T, stride, model->D, model->DP, d_i.as<int32_t>(), dw,
                                                 model->d_rows.as<float>(), model->d_gconsts.as<float>(),
                                                 model->d_pdf_offsets.as<int32_t>(), P, d_o.as<int32_t>(), nullptr, nullptr,
                                                 d_p.as<float>(), d_like.as<double>(), bad, d_l.as<float>());
  VB_CUDA(cudaGetLastError());
  if (R > 0) VB_CUDA(cudaMemcpy(post, d_p.p, (size_t)R * 4, cudaMemcpyDeviceToHost));
  if (loglikes) VB_CUDA(cudaMemcpy(loglikes, d_l.p, (size_t)T * 4, cudaMemcpyDeviceToHost));
  VB_TRY(count.end(0, &n_bad));
  if (n_bad) return fail(VBGPU_ERR_NUMERIC, "%llu frames had an invalid pdf-id or a NaN/Inf likelihood", n_bad);
  return 0;
}

}  // extern "C"
