// accum.cu — EM sufficient statistics from alignments: AccumAmDiagGmm::AccumulateForGmm[Twofeats]
// (gmm/mle-am-diag-gmm.cc:69-97) -> AccumDiagGmm::AccumulateFromDiag / AccumulateFromPosteriors
// (gmm/mle-diag-gmm.cc:171-204) -> DiagGmm::ComponentPosteriors (gmm/diag-gmm.cc:601-615) + ApplySoftMax
// (matrix/kaldi-vector.cc:852-859).
//
// Main path ("bucketed"): the frames of a call are counting-sorted by aligned pdf on the device (histogram, scan,
// scatter), then a CTA takes one (pdf, chunk of <= 128 of its frames): a warp per frame computes the posteriors (lanes split
// the pdf's Gaussians: one FP32 dot product each, the reference's arithmetic; warp softmax) into shared memory, and the
// CTA then forms  occ_m += gamma, mean_md += gamma*y_d, var_md += gamma*y_d^2  for the whole chunk in FP64 REGISTERS
// (gamma widened to double, y^2 formed in double, as the reference does) and flushes each sum with ONE
// red.global.add.f64 — 1/128 of the global atomics of the frame-at-a-time form, which was bound by them.
// Pdfs with more than 64 Gaussians take the frame-at-a-time kernel (acc_kernel: a warp owns a frame and adds straight
// into the global accumulators).
// The accumulator is ONE buffer [occ | mean | var | tot_like | tot_frames] so that the cross-GPU reduce is one
// all-reduce.
#include <algorithm>
#include <cfloat>
#include <cstdlib>

#include "common.h"

namespace {

constexpr int kWarps = 8;
constexpr int kMaxD = 128;

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

__global__ void __launch_bounds__(kWarps * 32) acc_kernel(const float *__restrict__ feats,
                                                          const float *__restrict__ feats2, int64_t T, int32_t stride,
                                                          int32_t D, int32_t DP, const int32_t *__restrict__ pdf_ids,
                                                          const float *__restrict__ weights,
                                                          const float *__restrict__ rows,  // [N][2*DP]
                                                          const float *__restrict__ gconsts,
                                                          const int32_t *__restrict__ pdf_offsets, int32_t P,
                                                          int32_t N, double *__restrict__ acc,
                                                          unsigned long long *bad, int32_t min_gauss) {
  // min_gauss > 0: only frames whose pdf has more than min_gauss Gaussians (the rest went through acc_bucket_kernel)
  __shared__ float s_x[kWarps][2 * kMaxD];   // x | x^2 of the warp's frame (posterior features)
  __shared__ float s_post[kWarps][32];
  __shared__ double s_like[kWarps], s_cnt[kWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double *occ = acc, *mean = acc + N, *var = acc + N + (size_t)N * D;
  double like = 0.0, cnt = 0.0;
  unsigned long long nbad = 0;

  for (int64_t t = (int64_t)blockIdx.x * kWarps + warp; t < T; t += (int64_t)gridDim.x * kWarps) {
    const int p = pdf_ids[t];
    if (p < 0 || p >= P) {  // invalid alignment entry: counted as an error, frame skipped
      if (lane == 0 && min_gauss == 0) nbad++;  // (the bucketed path counts them itself)
      continue;
    }
    if (min_gauss > 0 && pdf_offsets[p + 1] - pdf_offsets[p] <= min_gauss) continue;
    const float w = weights ? weights[t] : 1.0f;
    const float *xr = feats + t * stride;
    for (int d = lane; d < D; d += 32) {
      const float v = xr[d];
      s_x[warp][d] = v;
      s_x[warp][kMaxD + d] = v * v;
    }
    __syncwarp();
    const int g0 = pdf_offsets[p], M = pdf_offsets[p + 1] - g0;
    const float *yr = (feats2 ? feats2 : feats) + t * stride;

    // pass over the Gaussians in chunks of 32 (lane = Gaussian): online max / sum across chunks
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
      const float cmax = warp_max(ll);
      const float nmax = fmaxf(run_max, cmax);
      const float e = (m < M && nmax > -INFINITY) ? __expf(ll - nmax) : 0.0f;
      const float csum = warp_sumf(e);
      run_sum = (run_max > -INFINITY ? run_sum * __expf(run_max - nmax) : 0.0f) + csum;
      run_max = nmax;
    }
    const float log_like = run_max + __logf(run_sum);  // ApplySoftMax returns max + Log(sum)
    if (!(fabsf(log_like) <= FLT_MAX)) {               // diag-gmm.cc:609-610 raises KALDI_ERR
      if (lane == 0) nbad++;
      __syncwarp();
      continue;
    }
    const float inv_sum = 1.0f / run_sum;

    // second pass: posteriors chunk by chunk, then lanes switch to dimensions for the FP64 accumulation
    for (int c0 = 0; c0 < M; c0 += 32) {
      const int m = c0 + lane;
      float post = 0.0f;
      if (m < M) {
        const float *r = rows + (size_t)(g0 + m) * (2 * DP);
        float a = 0.0f, b = 0.0f;
        for (int d = 0; d < D; d++) a = fmaf(r[d], s_x[warp][d], a);
        for (int d = 0; d < D; d++) b = fmaf(r[DP + d], s_x[warp][kMaxD + d], b);
        const float ll = (gconsts[g0 + m] + a) + b;
        post = __expf(ll - run_max) * inv_sum * w;  // Exp(x-max), Scale(1/sum), Scale(frame_posterior)
        atomicAdd(&occ[g0 + m], (double)post);      // occupancy_.AddVec(1.0, post_d)
      }
      s_post[warp][lane] = post;
      __syncwarp();
      const int mc = min(32, M - c0);
      for (int d = lane; d < D; d += 32) {
        const double yd = (double)yr[d], yd2 = yd * yd;  // data_d.ApplyPow(2.0) in double
        for (int k = 0; k < mc; k++) {
          const double g = (double)s_post[warp][k];
          if (g != 0.0) {
            atomicAdd(&mean[(size_t)(g0 + c0 + k) * D + d], g * yd);
            atomicAdd(&var[(size_t)(g0 + c0 + k) * D + d], g * yd2);
          }
        }
      }
      __syncwarp();
    }
    if (lane == 0) {
      like += (double)(log_like * w);  // total_log_like_ += log_like * weight (float product)
      cnt += (double)w;
    }
  }
  if (lane == 0) {
    s_like[warp] = like;
    s_cnt[warp] = cnt;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double l = 0.0, c = 0.0;
    for (int i = 0; i < kWarps; i++) {
      l += s_like[i];
      c += s_cnt[i];
    }
    const size_t tail = (size_t)N + 2 * (size_t)N * D;
    if (c != 0.0 || l != 0.0) {
      atomicAdd(&acc[tail], l);
      atomicAdd(&acc[tail + 1], c);
    }
  }
  if (nbad) atomicAdd(bad, nbad);
}

// ---- bucketed path ----------------------------------------------------------------------------------------------------
constexpr int kChunk = vb::kSortChunk;  // frames of one pdf per work unit
constexpr int kMaxM = 64;     // Gaussians per pdf served by the bucketed kernel
// workspace (int32): count[P+1] | start[P+2] | cursor[P+1] | unit_off[P+2] | order[T]      (bin P = invalid pdf ids)

__global__ void acc_hist_kernel(const int32_t *__restrict__ pdf_ids, int64_t T, int32_t P, int32_t *__restrict__ count) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < T; t += (int64_t)gridDim.x * blockDim.x) {
    const int p = pdf_ids[t];
    atomicAdd(&count[(p < 0 || p >= P) ? P : p], 1);
  }
}

// One block: exclusive scans of the counts (-> start, cursor) and of the units per pdf (-> unit_off).  pdf_offsets == NULL
// (the LDA statistics): every bin gets units.
__global__ void acc_scan_kernel(const int32_t *__restrict__ count, const int32_t *__restrict__ pdf_offsets, int32_t P,
                                int32_t *__restrict__ start, int32_t *__restrict__ cursor, int32_t *__restrict__ unit_off,
                                unsigned long long *bad) {
  __shared__ int32_t s_a[1024], s_b[1024];
  __shared__ int32_t base_a, base_b;
  if (threadIdx.x == 0) base_a = 0, base_b = 0;
  __syncthreads();
  for (int p0 = 0; p0 <= P; p0 += 1024) {
    const int p = p0 + threadIdx.x;
    int c = 0, u = 0;
    if (p <= P) {
      c = count[p];
      if (p < P && (!pdf_offsets || pdf_offsets[p + 1] - pdf_offsets[p] <= kMaxM)) u = (c + kChunk - 1) / kChunk;
    }
    s_a[threadIdx.x] = c;
    s_b[threadIdx.x] = u;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {  // Hillis-Steele inclusive scan
      int va = 0, vb = 0;
      if ((int)threadIdx.x >= o) va = s_a[threadIdx.x - o], vb = s_b[threadIdx.x - o];
      __syncthreads();
      s_a[threadIdx.x] += va;
      s_b[threadIdx.x] += vb;
      __syncthreads();
    }
    if (p <= P) {
      start[p] = base_a + s_a[threadIdx.x] - c;
      cursor[p] = base_a + s_a[threadIdx.x] - c;
      unit_off[p] = base_b + s_b[threadIdx.x] - u;
    }
    __syncthreads();
    if (threadIdx.x == 1023) base_a += s_a[1023], base_b += s_b[1023];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    start[P + 1] = base_a;
    unit_off[P + 1] = base_b;  // total units
    if (count[P] > 0) atomicAdd(bad, (unsigned long long)count[P]);  // invalid alignment entries: an error, frames skipped
  }
}

__global__ void acc_scatter_kernel(const int32_t *__restrict__ pdf_ids, int64_t T, int32_t P, int32_t *__restrict__ cursor,
                                   int32_t *__restrict__ order) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < T; t += (int64_t)gridDim.x * blockDim.x) {
    const int p = pdf_ids[t];
    order[atomicAdd(&cursor[(p < 0 || p >= P) ? P : p], 1)] = (int32_t)t;
  }
}

// dynamic shared memory (floats): x[kChunk][DY] posterior features | y[kChunk][DY] statistics features (aliases x
// unless feats2) | r[2*D][kMP] the pdf's model rows, transposed | g[kChunk][kMP] log-likelihoods, then posteriors
constexpr int kMP = kMaxM + 1;  // odd pitch: the transposing stores of the model rows are conflict-free
__global__ void __launch_bounds__(kWarps * 32) acc_bucket_kernel(
    const float *__restrict__ feats, const float *__restrict__ feats2, int32_t stride, int32_t D, int32_t DP, int32_t DY,
    const float *__restrict__ weights, const float *__restrict__ rows, const float *__restrict__ gconsts,
    const int32_t *__restrict__ pdf_offsets, int32_t P, int32_t N, const int32_t *__restrict__ start,
    const int32_t *__restrict__ unit_off, const int32_t *__restrict__ order, double *__restrict__ acc,
    unsigned long long *bad, float *__restrict__ ab_out, int32_t ab_pitch, float *__restrict__ cnt_out,
    double *__restrict__ like_out) {
  // ab_out != NULL: "posterior mode" for the fMLLR statistics (fmllr.cu): instead of the EM sums, every frame gets
  // a = sum_m gamma_m means_invvars_m, b = sum_m gamma_m inv_vars_m (FP32) and count = sum_m gamma_m, and like_out the
  // unweighted sum of the frames' log-likelihoods (FmllrDiagGmmAccs::AccumulateFromPosteriors, fmllr-diag-gmm.cc:30-45).
  extern __shared__ __align__(16) float smem_f[];
  float *s_x = smem_f, *s_y = feats2 ? s_x + kChunk * DY : s_x, *s_r = s_y + kChunk * DY, *s_g = s_r + 2 * D * kMP;
  __shared__ int32_t s_pdf;
  __shared__ double s_like[kWarps], s_cnt[kWarps];
  constexpr int kThreads = kWarps * 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double *occ = acc, *mean = acc + N, *var = acc + N + (size_t)N * D;
  double like = 0.0, cnt = 0.0;
  unsigned long long nbad = 0;
  const int n_units = unit_off[P + 1];
  // 16-byte row loads: rows aligned and long enough to read the last quarter whole
  const bool vec_rows = DY % 4 == 0 && stride % 4 == 0 && stride >= (D + 3) / 4 * 4 &&
                        (reinterpret_cast<uintptr_t>(feats) & 15) == 0 &&
                        (feats2 == nullptr || (reinterpret_cast<uintptr_t>(feats2) & 15) == 0);

  for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
    if (threadIdx.x == 0) {  // the pdf of unit u: last p with unit_off[p] <= u
      int lo = 0, hi = P;
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (unit_off[mid] <= u) lo = mid;
        else hi = mid;
      }
      s_pdf = lo;
    }
    __syncthreads();
    const int p = s_pdf;
    const int f0 = start[p] + (u - unit_off[p]) * kChunk, n = min(kChunk, start[p + 1] - f0);
    const int g0 = pdf_offsets[p], M = pdf_offsets[p + 1] - g0;

    // ---- stage the chunk's feature rows (gathered through the sorted order) and the pdf's model rows ----
    if (vec_rows) {
      // rows as float4: a thread owns one quarter-row slot (row, q) per pass, its `order` entry and row are loaded once
      // and the passes are independent, so several gathers are in flight per thread
      const int qpr = DY / 4;
      for (int idx = threadIdx.x; idx < n * qpr; idx += kThreads) {
        const int i = idx / qpr, q = idx - i * qpr;
        const int64_t t = order[f0 + i];
        float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (4 * q < D) v = *reinterpret_cast<const float4 *>(feats + t * stride + 4 * q);
        if (4 * q + 1 >= D) v.y = 0.0f;
        if (4 * q + 2 >= D) v.z = 0.0f;
        if (4 * q + 3 >= D) v.w = 0.0f;
        *reinterpret_cast<float4 *>(s_x + i * DY + 4 * q) = v;
        if (feats2) {
          float4 y = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
          if (4 * q < D) y = *reinterpret_cast<const float4 *>(feats2 + t * stride + 4 * q);
          if (4 * q + 1 >= D) y.y = 0.0f;
          if (4 * q + 2 >= D) y.z = 0.0f;
          if (4 * q + 3 >= D) y.w = 0.0f;
          *reinterpret_cast<float4 *>(s_y + i * DY + 4 * q) = y;
        }
      }
    } else {
      for (int idx = threadIdx.x; idx < n * DY; idx += kThreads) {
        const int i = idx / DY, d = idx - i * DY;
        const int64_t t = order[f0 + i];
        s_x[idx] = d < D ? feats[t * stride + d] : 0.0f;
        if (feats2) s_y[idx] = d < D ? feats2[t * stride + d] : 0.0f;
      }
    }
    for (int idx = threadIdx.x; idx < M * 2 * DP; idx += kThreads) {
      const int m = idx / (2 * DP), j = idx - m * 2 * DP, d = j < DP ? j : j - DP;
      if (d < D) s_r[(j < DP ? d : D + d) * kMP + m] = rows[(size_t)g0 * 2 * DP + idx];
    }
    __syncthreads();

    // ---- log-likelihoods: a thread per (frame, Gaussian): gconst + means_invvars.x - 0.5 inv_vars.x^2, FP32 FMAs ----
    // A thread takes one Gaussian and FOUR frames: a model value is read once per four products and the frames' rows
    // arrive as float4; every (frame, Gaussian) sum still runs over d in order, so the values are those of the
    // one-frame form.  (Rows past n hold an earlier chunk's features: computed, not stored.)
    for (int idx = threadIdx.x; idx < ((n + 3) >> 2) * M; idx += kThreads) {
      const int q = idx / M, m = idx - q * M;
      const float *x0 = s_x + 4 * q * DY;
      float a[4] = {0.0f, 0.0f, 0.0f, 0.0f}, b[4] = {0.0f, 0.0f, 0.0f, 0.0f};
      int d = 0;
      for (; d + 4 <= D; d += 4) {
        const float ra0 = s_r[d * kMP + m], ra1 = s_r[(d + 1) * kMP + m], ra2 = s_r[(d + 2) * kMP + m], ra3 = s_r[(d + 3) * kMP + m];
        const float rb0 = s_r[(D + d) * kMP + m], rb1 = s_r[(D + d + 1) * kMP + m], rb2 = s_r[(D + d + 2) * kMP + m],
                    rb3 = s_r[(D + d + 3) * kMP + m];
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const float4 x = *reinterpret_cast<const float4 *>(x0 + k * DY + d);
          a[k] = fmaf(ra0, x.x, a[k]);
          a[k] = fmaf(ra1, x.y, a[k]);
          a[k] = fmaf(ra2, x.z, a[k]);
          a[k] = fmaf(ra3, x.w, a[k]);
          b[k] = fmaf(rb0, x.x * x.x, b[k]);
          b[k] = fmaf(rb1, x.y * x.y, b[k]);
          b[k] = fmaf(rb2, x.z * x.z, b[k]);
          b[k] = fmaf(rb3, x.w * x.w, b[k]);
        }
      }
      for (; d < D; d++) {
        const float ra = s_r[d * kMP + m], rb = s_r[(D + d) * kMP + m];
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const float x = x0[k * DY + d];
          a[k] = fmaf(ra, x, a[k]);
          b[k] = fmaf(rb, x * x, b[k]);
        }
      }
      const float gc = gconsts[g0 + m];
#pragma unroll
      for (int k = 0; k < 4; k++)
        if (4 * q + k < n) s_g[(4 * q + k) * kMP + m] = (gc + a[k]) + b[k];
    }
    __syncthreads();

    // ---- softmax per frame (ApplySoftMax, kaldi-vector.cc:852-859: max, sequential float sum), times the frame weight ----
    for (int i = threadIdx.x; i < n; i += kThreads) {
      float *g = s_g + i * kMP;
      const float w = weights ? weights[order[f0 + i]] : 1.0f;
      float mx = -INFINITY, sum = 0.0f;
      for (int m = 0; m < M; m++) mx = fmaxf(mx, g[m]);
      for (int m = 0; m < M; m++) {
        const float e = mx > -INFINITY ? __expf(g[m] - mx) : 0.0f;
        g[m] = e;
        sum += e;
      }
      const float log_like = mx + __logf(sum);       // ApplySoftMax returns max + Log(sum)
      const bool ok = fabsf(log_like) <= FLT_MAX;   // diag-gmm.cc:609-610 raises KALDI_ERR otherwise
      const float inv_sum = 1.0f / sum;
      for (int m = 0; m < M; m++) g[m] = ok ? g[m] * inv_sum * w : 0.0f;  // Scale(1/sum), Scale(frame_posterior)
      if (ok) {
        like += ab_out ? (double)log_like : (double)(log_like * w);  // total_log_like_ += log_like * weight (float product)
        cnt += (double)w;
      } else {
        nbad++;  // the frame adds nothing
      }
    }
    __syncthreads();

    if (ab_out) {  // ---- posterior mode: a thread per (frame, dimension) ----
      for (int idx = threadIdx.x; idx < n * D; idx += kThreads) {
        const int i = idx / D, d = idx - i * D;
        const float *g = s_g + i * kMP;
        float a = 0.0f, b = 0.0f;
        for (int m = 0; m < M; m++) {
          a = fmaf(g[m], s_r[d * kMP + m], a);
          b = fmaf(g[m], -2.0f * s_r[(D + d) * kMP + m], b);  // the rows hold -0.5 inv_vars
        }
        float *o = ab_out + (int64_t)order[f0 + i] * (2 * ab_pitch);
        o[d] = a;
        o[ab_pitch + d] = b;
      }
      for (int i = threadIdx.x; i < n; i += kThreads) {
        const float *g = s_g + i * kMP;
        double c = 0.0;
        for (int m = 0; m < M; m++) c += (double)g[m];  // posterior.Sum(): double sum handed back as float
        cnt_out[order[f0 + i]] = (float)c;
      }
      __syncthreads();
      continue;
    }
    // ---- statistics: a thread per (Gaussian, dimension): FP64 sums over the chunk, one atomic each ----
    // (two adjacent dimensions per thread: the posterior is converted once for both, the features arrive as float2, and a
    // 10-Gaussian pdf at D = 39 fits one round of the CTA; every sum runs over the frames in order as before)
    const int DH = (D + 1) >> 1;
    for (int idx = threadIdx.x; idx < M * DH; idx += kThreads) {
      const int k = idx / DH, d = 2 * (idx - k * DH);
      double m1a = 0.0, m2a = 0.0, m1b = 0.0, m2b = 0.0;
      for (int i = 0; i < n; i++) {
        const double g = (double)s_g[i * kMP + k];
        const float2 yy = *reinterpret_cast<const float2 *>(s_y + i * DY + d);  // (DY is even: d + 1 < DY, zero past D)
        const double ya = (double)yy.x, yb = (double)yy.y;
        m1a += g * ya;
        m2a += g * (ya * ya);
        m1b += g * yb;
        m2b += g * (yb * yb);
      }
      atomicAdd(&mean[(size_t)(g0 + k) * D + d], m1a);
      atomicAdd(&var[(size_t)(g0 + k) * D + d], m2a);
      if (d + 1 < D) {
        atomicAdd(&mean[(size_t)(g0 + k) * D + d + 1], m1b);
        atomicAdd(&var[(size_t)(g0 + k) * D + d + 1], m2b);
      }
    }
    for (int k = threadIdx.x; k < M; k += kThreads) {
      double o = 0.0;
      for (int i = 0; i < n; i++) o += (double)s_g[i * kMP + k];
      atomicAdd(&occ[g0 + k], o);
    }
    __syncthreads();
  }
  for (int o = 16; o > 0; o >>= 1) {
    like += __shfl_xor_sync(0xffffffffu, like, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if (lane == 0) {
    s_like[warp] = like;
    s_cnt[warp] = cnt;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double l = 0.0, c = 0.0;
    for (int i = 0; i < kWarps; i++) {
      l += s_like[i];
      c += s_cnt[i];
    }
    const size_t tail = (size_t)N + 2 * (size_t)N * D;
    if (like_out) {
      if (l != 0.0) atomicAdd(like_out, l);
    } else if (c != 0.0 || l != 0.0) {
      atomicAdd(&acc[tail], l);
      atomicAdd(&acc[tail + 1], c);
    }
  }
  if (nbad) atomicAdd(bad, nbad);
}

__global__ void axpy_kernel(double *__restrict__ dst, const double *__restrict__ src, double scale, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    dst[i] += scale * src[i];
}

}  // namespace

namespace vb {

int bin_sort_launch(const int32_t *d_ids, int64_t T, int32_t P, const int32_t *d_pdf_offsets, int device, DevBuf *work,
                    unsigned long long *bad, cudaStream_t s, BinSort *out) {
  const size_t n_int = (size_t)(P + 1) + (P + 2) + (P + 1) + (P + 2) + (size_t)T;
  VB_TRY(work->reserve(n_int * 4));
  int32_t *count = work->as<int32_t>(), *start = count + (P + 1), *cursor = start + (P + 2), *unit_off = cursor + (P + 1),
          *order = unit_off + (P + 2);
  VB_CUDA(cudaMemsetAsync(count, 0, (size_t)(P + 1) * 4, s));
  const int g1 = (int)std::min<int64_t>((T + 255) / 256, (int64_t)num_sms(device) * 16);
  acc_hist_kernel<<<g1, 256, 0, s>>>(d_ids, T, P, count);
  acc_scan_kernel<<<1, 1024, 0, s>>>(count, d_pdf_offsets, P, start, cursor, unit_off, bad);
  acc_scatter_kernel<<<g1, 256, 0, s>>>(d_ids, T, P, cursor, order);
  VB_CUDA(cudaGetLastError());
  *out = BinSort{start, unit_off, order};
  return 0;
}

int acc_launch(vbgpu_acc_t h, const float *d_feats, const float *d_feats2, int64_t T, int32_t stride,
               const int32_t *d_ids, const float *d_w, cudaStream_t s) {
  if (T == 0) return 0;
  vbgpu_gmm_t g = h->model;
  if (g->D > kMaxD) return fail(VBGPU_ERR_INVALID, "feature dim %d > %d", g->D, kMaxD);
  if (T >= (int64_t)1 << 31) return fail(VBGPU_ERR_INVALID, "more than 2^31 frames in one call");
  const int P = g->P, sms = num_sms(h->device);
  const int DY = (g->D + 3) / 4 * 4;
  const size_t smem = ((size_t)kChunk * DY * (d_feats2 ? 2 : 1) + (size_t)2 * g->D * kMP + (size_t)kChunk * kMP) * 4;
  // the bucketed kernel stages a chunk of frames and the pdf's rows in shared memory: shapes that do not fit take the
  // frame-wise kernel instead of failing at launch
  const bool bucket = getenv("VBGPU_ACC_FRAMEWISE") == nullptr && smem <= 200 * 1024;
  if (bucket) {
    // counting sort of the frames by pdf, then (pdf, chunk) work units
    BinSort bs;
    VB_TRY(bin_sort_launch(d_ids, T, P, g->d_pdf_offsets.as<int32_t>(), h->device, &h->d_work,
                           g->d_bad.as<unsigned long long>(), s, &bs));
    if (!h->bucket_attr_set) {
      VB_CUDA(cudaFuncSetAttribute(acc_bucket_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      h->bucket_attr_set = true;
    }
    const int64_t max_units = (int64_t)P + T / kChunk + 1;
    const int g2 = (int)std::min<int64_t>(max_units, (int64_t)sms * 3);
    acc_bucket_kernel<<<g2, kWarps * 32, smem, s>>>(d_feats, d_feats2, stride, g->D, g->DP, DY, d_w, g->d_rows.as<float>(),
                                                    g->d_gconsts.as<float>(), g->d_pdf_offsets.as<int32_t>(), P, g->N, bs.start,
                                                    bs.unit_off, bs.order, h->d_acc.as<double>(),
                                                    g->d_bad.as<unsigned long long>(), nullptr, 0, nullptr, nullptr);
    VB_CUDA(cudaGetLastError());
    if (g->max_pdf_size <= kMaxM) return 0;
  }
  int64_t blocks = (T + kWarps - 1) / kWarps;
  int64_t cap = (int64_t)sms * 8;
  int grid = (int)(blocks < cap ? blocks : cap);
  acc_kernel<<<grid, kWarps * 32, 0, s>>>(d_feats, d_feats2, T, stride, g->D, g->DP, d_ids, d_w, g->d_rows.as<float>(),
                                          g->d_gconsts.as<float>(), g->d_pdf_offsets.as<int32_t>(), g->P, g->N,
                                          h->d_acc.as<double>(), g->d_bad.as<unsigned long long>(), bucket ? kMaxM : 0);
  VB_CUDA(cudaGetLastError());
  return 0;
}

// Posterior mode of the bucketed kernel for the fMLLR statistics: per-frame a, b (pitch ab_pitch floats each) and count
// for every frame whose pdf has at most kMaxM Gaussians; returns that bound so that the caller serves the rest.
int acc_posterior_ab_launch(vbgpu_gmm_t g, DevBuf *work, const float *d_feats, int64_t T, int32_t stride,
                            const int32_t *d_ids, const float *d_w, float *d_ab, int32_t ab_pitch, float *d_cnt,
                            double *d_like, int32_t *max_gauss_served, cudaStream_t s) {
  const int P = g->P, sms = num_sms(g->device);
  BinSort bs;
  VB_TRY(bin_sort_launch(d_ids, T, P, g->d_pdf_offsets.as<int32_t>(), g->device, work, g->d_bad.as<unsigned long long>(),
                         s, &bs));
  const int DY = (g->D + 3) / 4 * 4;
  const size_t smem = ((size_t)kChunk * DY + (size_t)2 * g->D * kMP + (size_t)kChunk * kMP) * 4;
  // (per device: set on every call — a process may drive several GPUs, and the call costs microseconds)
  VB_CUDA(cudaFuncSetAttribute(acc_bucket_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  const int64_t max_units = (int64_t)P + T / kChunk + 1;
  const int g2 = (int)std::min<int64_t>(max_units, (int64_t)sms * 3);
  acc_bucket_kernel<<<g2, kWarps * 32, smem, s>>>(d_feats, nullptr, stride, g->D, g->DP, DY, d_w, g->d_rows.as<float>(),
                                                  g->d_gconsts.as<float>(), g->d_pdf_offsets.as<int32_t>(), P, g->N, bs.start,
                                                  bs.unit_off, bs.order, nullptr, g->d_bad.as<unsigned long long>(), d_ab, ab_pitch,
                                                  d_cnt, d_like);
  VB_CUDA(cudaGetLastError());
  *max_gauss_served = kMaxM;
  return 0;
}

int acc_axpy(double *d_dst, const double *d_src, double scale, int64_t n, cudaStream_t s) {
  if (n == 0) return 0;
  int grid = (int)((n + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  axpy_kernel<<<grid, 256, 0, s>>>(d_dst, d_src, scale, n);
  VB_CUDA(cudaGetLastError());
  return 0;
}

// Transition accumulators (TransitionModel::Accumulate(1.0, tid, &transition_accs), gmm-acc-stats-ali.cpp:92): a histogram
// of the alignment's transition-ids.  Alignments are runs of self-loops: a thread walks 64 consecutive frames and emits one
// FP64 atomic per run.
__global__ void __launch_bounds__(256) acc_transitions_kernel(double *__restrict__ trans, int32_t n_trans,
                                                              const int32_t *__restrict__ tids, int64_t T,
                                                              unsigned long long *bad) {
  const int64_t t0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 64;
  if (t0 >= T) return;
  const int64_t t1 = t0 + 64 < T ? t0 + 64 : T;
  int32_t cur = tids[t0];
  double run = 0.0;
  unsigned long long nbad = 0;
  for (int64_t t = t0; t < t1; t++) {
    const int32_t id = tids[t];
    if (id != cur) {
      if (cur >= 1 && cur < n_trans) atomicAdd(trans + cur, run);
      else nbad += (unsigned long long)run;
      cur = id;
      run = 0.0;
    }
    run += 1.0;
  }
  if (cur >= 1 && cur < n_trans) atomicAdd(trans + cur, run);
  else nbad += (unsigned long long)run;
  if (nbad) atomicAdd(bad, nbad);
}

int acc_transitions_launch(double *d_trans, int32_t n_trans, const int32_t *d_tids, int64_t T, unsigned long long *bad,
                           cudaStream_t s) {
  if (T == 0) return 0;
  const int64_t threads = (T + 63) / 64;
  acc_transitions_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(d_trans, n_trans, d_tids, T, bad);
  VB_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace vb
