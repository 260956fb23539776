// lda.cu — LDA class statistics: LdaEstimate::Accumulate (transform/lda-estimate.cc) as acc-lda drives it, one
// (class, weight) per frame from ali-to-post | weight-silence-post.  For every frame t with class c_t and weight w_t != 0:
//     zero[c_t] += w_t        first[c_t][:] += w_t x_t        second += w_t x_t x_t^T  (packed lower triangle, SpMatrix order)
// All sums are FP64, as the reference keeps them: x is widened to double before any product (a float x float product is
// exact in double), so the results differ from the reference's only by the order of the FP64 additions.
//
// Three steps:
//   sort             frames counting-sorted by class (bin_sort_launch, shared with the EM statistics in accum.cu); invalid
//                    class ids land in a bin without work and are counted.
//   lda_class_kernel a CTA per (class, chunk of <= 128 of its frames): a thread per dimension sums w x over the chunk in a
//                    register and flushes it with ONE FP64 atomic, thread 0 likewise for the weights.
//   lda_tri_kernel   second = X^T diag(w) X over the packed triangle: a CTA owns a chunk of frames (staged 16 at a time in
//                    shared memory as double rows w x and x, the next 16 copied with cp.async meanwhile) and up to 128 8 x 8
//                    blocks of the lower triangle, one block per thread held in 64 FP64 registers; FP64 FMAs, one
//                    red.global.add.f64 per element per chunk.
// Frames of weight exactly 0 are skipped (acc-lda never calls Accumulate for them), so non-finite features there are
// harmless; frames with an invalid class id add nothing to any statistic.
#include <cuda_pipeline.h>

#include <algorithm>

#include "common.h"

namespace {

constexpr int kClassThreads = 128;
constexpr int kTB = 8;            // thread tile: kTB x kTB block of the D x D square
constexpr int kFT = 16;           // frames per shared-memory stage of the triangle kernel
constexpr int kTriThreads = 128;  // triangle blocks per CTA (larger D: more CTAs along y)

__global__ void __launch_bounds__(kClassThreads) lda_class_kernel(const float *__restrict__ feats, int32_t stride,
                                                                  int32_t D, int32_t C, const float *__restrict__ weights,
                                                                  const int32_t *__restrict__ start,
                                                                  const int32_t *__restrict__ unit_off,
                                                                  const int32_t *__restrict__ order,
                                                                  double *__restrict__ zero, double *__restrict__ first) {
  __shared__ int32_t s_t[vb::kSortChunk];
  __shared__ float s_w[vb::kSortChunk];
  __shared__ int32_t s_c;
  const int n_units = unit_off[C + 1];
  for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
    if (threadIdx.x == 0) {  // the class of unit u: last c with unit_off[c] <= u
      int lo = 0, hi = C;
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (unit_off[mid] <= u) lo = mid;
        else hi = mid;
      }
      s_c = lo;
    }
    __syncthreads();
    const int c = s_c;
    const int f0 = start[c] + (u - unit_off[c]) * vb::kSortChunk, n = min(vb::kSortChunk, start[c + 1] - f0);
    for (int i = threadIdx.x; i < n; i += kClassThreads) {
      const int t = order[f0 + i];
      s_t[i] = t;
      s_w[i] = weights ? weights[t] : 1.0f;
    }
    __syncthreads();
    for (int d = threadIdx.x; d < D; d += kClassThreads) {
      double acc = 0.0;
#pragma unroll 4
      for (int i = 0; i < n; i++) {
        const float w = s_w[i];
        if (w != 0.0f) acc += (double)w * (double)feats[(int64_t)s_t[i] * stride + d];
      }
      atomicAdd(&first[(size_t)c * D + d], acc);
    }
    if (threadIdx.x == 0) {
      double z = 0.0;
      for (int i = 0; i < n; i++) z += (double)s_w[i];
      atomicAdd(&zero[c], z);
    }
    __syncthreads();
  }
}

// dynamic shared memory: a[kFT][DP] = w x | b[kFT][DP] = x (doubles; zero for skipped frames and past D, DP = 8 ceil(D/8)),
// then raw[2][kFT][DP] floats: the rows of the next stage, copied with cp.async while the current stage is computed
__global__ void __launch_bounds__(kTriThreads) lda_tri_kernel(const float *__restrict__ feats, int64_t T, int32_t stride,
                                                              int32_t D, int32_t C, const int32_t *__restrict__ ids,
                                                              const float *__restrict__ weights, int64_t chunk,
                                                              int32_t n_tiles, double *__restrict__ second) {
  extern __shared__ __align__(16) double smem_d[];
  __shared__ int32_t s_id[2][kFT];
  __shared__ float s_wt[2][kFT];
  const int DP = (D + kTB - 1) / kTB * kTB;
  double *s_a = smem_d, *s_b = smem_d + kFT * DP;
  float *s_raw = reinterpret_cast<float *>(smem_d + 2 * kFT * DP);
  // this thread's block (bi, bj), bi >= bj, numbered row by row: q = bi (bi + 1) / 2 + bj
  const int q = blockIdx.y * kTriThreads + threadIdx.x;
  const bool active = q < n_tiles;
  int bi = (int)((sqrtf(8.0f * q + 1.0f) - 1.0f) * 0.5f);
  while (bi * (bi + 1) / 2 > q) bi--;
  while ((bi + 1) * (bi + 2) / 2 <= q) bi++;
  const int bj = q - bi * (bi + 1) / 2;

  double acc[kTB][kTB];
#pragma unroll
  for (int i = 0; i < kTB; i++)
#pragma unroll
    for (int j = 0; j < kTB; j++) acc[i][j] = 0.0;

  const int64_t t0 = (int64_t)blockIdx.x * chunk, t1 = min(T, t0 + chunk);
  auto issue = [&](int64_t tb, int buf) {  // asynchronous copies of frames [tb, tb + kFT): rows, class ids, weights
    if (threadIdx.x < kFT && tb + threadIdx.x < t1) {
      __pipeline_memcpy_async(&s_id[buf][threadIdx.x], ids + tb + threadIdx.x, 4);
      if (weights) __pipeline_memcpy_async(&s_wt[buf][threadIdx.x], weights + tb + threadIdx.x, 4);
    }
    float *raw = s_raw + buf * kFT * DP;
    for (int idx = threadIdx.x; idx < kFT * DP; idx += blockDim.x) {
      const int k = idx / DP, d = idx - k * DP;
      if (d < D && tb + k < t1) __pipeline_memcpy_async(raw + idx, feats + (tb + k) * stride + d, 4);
    }
    __pipeline_commit();
  };
  if (t0 < t1) issue(t0, 0);
  int buf = 0;
  for (int64_t tb = t0; tb < t1; tb += kFT, buf ^= 1) {
    __pipeline_wait_prior(0);
    __syncthreads();  // stage tb has landed; the previous stage's products are done with s_a / s_b
    const float *raw = s_raw + buf * kFT * DP;
    for (int idx = threadIdx.x; idx < kFT * DP; idx += blockDim.x) {
      const int k = idx / DP, d = idx - k * DP;
      float w = 0.0f;  // 0: the frame is skipped (past the chunk, invalid class, weight 0)
      if (tb + k < t1) {
        const int c = s_id[buf][k];
        if (c >= 0 && c < C) w = weights ? s_wt[buf][k] : 1.0f;
      }
      double a = 0.0, b = 0.0;
      if (w != 0.0f && d < D) {
        b = (double)raw[idx];
        a = (double)w * b;
      }
      s_a[idx] = a;
      s_b[idx] = b;
    }
    __syncthreads();  // s_a / s_b ready; raw[buf] is free for the stage after next
    if (tb + kFT < t1) issue(tb + kFT, buf ^ 1);
    if (active) {
#pragma unroll 2
      for (int k = 0; k < kFT; k++) {
        double a[kTB], b[kTB];
        const double2 *pa = reinterpret_cast<const double2 *>(s_a + k * DP + kTB * bi);
        const double2 *pb = reinterpret_cast<const double2 *>(s_b + k * DP + kTB * bj);
#pragma unroll
        for (int v = 0; v < kTB / 2; v++) {
          const double2 x = pa[v], y = pb[v];
          a[2 * v] = x.x;
          a[2 * v + 1] = x.y;
          b[2 * v] = y.x;
          b[2 * v + 1] = y.y;
        }
#pragma unroll
        for (int i = 0; i < kTB; i++)
#pragma unroll
          for (int j = 0; j < kTB; j++) acc[i][j] = fma(a[i], b[j], acc[i][j]);
      }
    }
  }
  if (!active) return;
#pragma unroll
  for (int i = 0; i < kTB; i++) {
    const int gi = kTB * bi + i;
    if (gi >= D) break;
#pragma unroll
    for (int j = 0; j < kTB; j++) {
      const int gj = kTB * bj + j;
      if (gj <= gi) atomicAdd(&second[(size_t)gi * (gi + 1) / 2 + gj], acc[i][j]);
    }
  }
}

}  // namespace

namespace vb {

int lda_launch(vbgpu_lda_t h, const float *d_feats, int64_t T, int32_t stride, const int32_t *d_ids, const float *d_w,
               unsigned long long *bad, cudaStream_t s) {
  if (T == 0) return 0;
  if (T >= (int64_t)1 << 31) return fail(VBGPU_ERR_INVALID, "more than 2^31 frames in one call");
  const int C = h->C, D = h->D, sms = num_sms(h->device);
  double *zero = h->d_acc.as<double>(), *first = zero + C, *second = first + (size_t)C * D;

  BinSort bs;
  VB_TRY(bin_sort_launch(d_ids, T, C, nullptr, h->device, &h->d_work, bad, s, &bs));
  const int64_t max_units = (int64_t)C + T / kSortChunk + 1;
  const int g1 = (int)std::min<int64_t>(max_units, (int64_t)sms * 16);
  lda_class_kernel<<<g1, kClassThreads, 0, s>>>(d_feats, stride, D, C, d_w, bs.start, bs.unit_off, bs.order, zero, first);
  VB_CUDA(cudaGetLastError());

  const int B = (D + kTB - 1) / kTB, n_tiles = B * (B + 1) / 2;
  const int gy = (n_tiles + kTriThreads - 1) / kTriThreads;
  const int threads = std::min((n_tiles + 31) / 32 * 32, kTriThreads);
  const size_t smem = (size_t)2 * kFT * B * kTB * (sizeof(double) + sizeof(float));
  // (per device: set on every call — a process may drive several GPUs, and the call costs microseconds)
  VB_CUDA(cudaFuncSetAttribute(lda_tri_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // one resident wave of equal chunks: each CTA flushes its blocks once, so fewer, longer chunks mean fewer atomics, and a
  // second, partial wave would leave SMs idle
  int per_sm = 0;
  VB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lda_tri_kernel, threads, smem));
  const int64_t want = std::max<int64_t>(1, (int64_t)sms * std::max(per_sm, 1) / gy);
  int64_t chunk = (T + want - 1) / want;
  chunk = (chunk + kFT - 1) / kFT * kFT;
  const int64_t n_chunks = (T + chunk - 1) / chunk;
  lda_tri_kernel<<<dim3((unsigned)n_chunks, gy), threads, smem, s>>>(d_feats, T, stride, D, C, d_ids, d_w, chunk, n_tiles,
                                                                      second);
  VB_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace vb
