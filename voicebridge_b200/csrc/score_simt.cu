// score_simt.cu — FP32 SIMT dense scoring: loglikes[t][p] = LogSumExp_{m in pdf p}( gconst_m + miv_m.x_t - 0.5 iv_m.x_t^2 ).
//
// The bit-for-bit-closest restatement of the reference's arithmetic (DiagGmm::LogLikelihoods, gmm/diag-gmm.cc:528-543,
// behind DecodableAmDiagGmmUnmapped::LogLikelihoodZeroBased, gmm/decodable-am-diag-gmm.cc:28-72): FP32 FMAs, one
// dot product per (frame, Gaussian).  It is the parity anchor for the tensor-core kernel (score_tc.cu) and the path
// taken when a model does not fit that kernel's constraints.
//
// Mapping: a thread owns ONE frame (x and x^2 live in registers), a warp owns 32 frames, and walks a range of pdfs;
// model rows are read with warp-uniform 128-bit loads (one L1 wavefront for 32 frames).  Per-pdf results of 32 pdfs are
// staged in a 32x33 shared tile and written as 128-byte rows.
#include <cfloat>

#include "common.h"

namespace {

constexpr int kWarps = 8;

// Online log-sum-exp update (the reference takes max first, drops terms below max+log(FLT_EPSILON) and sums the rest in
// double, kaldi-vector.cc:757-775; dropped terms change the result by < M*1.2e-7 relative, far inside the 1e-3 budget).
__device__ __forceinline__ void lse_push(float v, float &mx, float &sum) {
  if (v > mx) {  // (mx == -inf: sum is 0 and __expf(-inf) = 0)
    sum = sum * __expf(mx - v) + 1.0f;
    mx = v;
  } else if (v > -INFINITY) {  // a zero-weight Gaussian (gconst = -inf, diag-gmm.cc:141-146) contributes nothing
    sum += __expf(v - mx);
  }
}

template <int DP4>  // row length in float4 (DP = 4*DP4 >= D)
__global__ void __launch_bounds__(kWarps * 32) score_simt_kernel(const float *__restrict__ feats, int64_t T,
                                                                 int32_t stride, int32_t D,
                                                                 const float4 *__restrict__ rows,  // [N][2*DP4]
                                                                 const float *__restrict__ gconsts,
                                                                 const int32_t *__restrict__ pdf_offsets, int32_t P,
                                                                 int32_t pdfs_per_cta, float *__restrict__ out,
                                                                 int32_t out_stride, unsigned long long *bad) {
  constexpr int DP = 4 * DP4;
  __shared__ float tile[kWarps][32][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t t = ((int64_t)blockIdx.x * kWarps + warp) * 32 + lane;
  const int64_t t_warp0 = t - lane;
  const bool live = t < T;

  float x[DP], xs[DP];
#pragma unroll
  for (int d = 0; d < DP; d++) {
    const float v = (live && d < D) ? feats[t * stride + d] : 0.0f;
    x[d] = v;
    xs[d] = v * v;  // data_sq.ApplyPow(2.0)
  }

  const int p_begin = blockIdx.y * pdfs_per_cta;
  const int p_end = min(P, p_begin + pdfs_per_cta);
  unsigned long long nbad = 0;
  for (int p0 = p_begin; p0 < p_end; p0 += 32) {
    const int np = min(32, p_end - p0);
    for (int pi = 0; pi < np; pi++) {
      const int g0 = pdf_offsets[p0 + pi], g1 = pdf_offsets[p0 + pi + 1];
      float mx = -INFINITY, sum = 0.0f;
      for (int g = g0; g < g1; g++) {
        const float4 *r = rows + (size_t)g * (2 * DP4);
        float a = 0.0f, b = 0.0f;
#pragma unroll
        for (int q = 0; q < DP4; q++) {
          const float4 m = __ldg(r + q);
          a = fmaf(m.x, x[4 * q + 0], a);
          a = fmaf(m.y, x[4 * q + 1], a);
          a = fmaf(m.z, x[4 * q + 2], a);
          a = fmaf(m.w, x[4 * q + 3], a);
        }
#pragma unroll
        for (int q = 0; q < DP4; q++) {
          const float4 m = __ldg(r + DP4 + q);  // -0.5 * inv_vars
          b = fmaf(m.x, xs[4 * q + 0], b);
          b = fmaf(m.y, xs[4 * q + 1], b);
          b = fmaf(m.z, xs[4 * q + 2], b);
          b = fmaf(m.w, xs[4 * q + 3], b);
        }
        const float ll = (__ldg(gconsts + g) + a) + b;  // gconst, += sgemv(miv), += sgemv(-0.5 iv)
        lse_push(ll, mx, sum);
      }
      const float res = (g1 > g0) ? mx + __logf(sum) : -INFINITY;
      if (live && !(fabsf(res) <= FLT_MAX)) nbad++;
      tile[warp][lane][pi] = res;
    }
    __syncwarp();
    // coalesced store: row r of the tile = frame t_warp0 + r, columns p0 .. p0+np
    for (int r = 0; r < 32; r++) {
      const int64_t tt = t_warp0 + r;
      if (tt < T && lane < np) out[tt * out_stride + p0 + lane] = tile[warp][r][lane];
    }
    __syncwarp();
  }
  if (nbad) atomicAdd(bad, nbad);
}

}  // namespace

namespace vb {

int score_simt_launch(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, float *d_ll, int32_t ll_stride,
                      unsigned long long *bad, cudaStream_t s) {
  if (T == 0) return 0;
  const int64_t frame_ctas = (T + kWarps * 32 - 1) / (kWarps * 32);
  // split the pdfs over grid.y so that small batches still fill the GPU (>= 2 waves of 148 SMs x 2 CTAs)
  int64_t want = 4LL * num_sms(h->device);
  int ysplit = (int)((want + frame_ctas - 1) / frame_ctas);
  int max_split = (h->P + 31) / 32;
  if (ysplit > max_split) ysplit = max_split;
  if (ysplit < 1) ysplit = 1;
  int pdfs_per_cta = ((h->P + ysplit - 1) / ysplit + 31) / 32 * 32;
  ysplit = (h->P + pdfs_per_cta - 1) / pdfs_per_cta;
  if (frame_ctas > 2147483647LL) return fail(VBGPU_ERR_INVALID, "too many frames in one call");
  dim3 grid((unsigned)frame_ctas, (unsigned)ysplit);
  const float4 *rows = h->d_rows.as<float4>();
  const float *gc = h->d_gconsts.as<float>();
  const int32_t *po = h->d_pdf_offsets.as<int32_t>();
#define VB_LAUNCH(DP4)                                                                                          \
  score_simt_kernel<DP4><<<grid, kWarps * 32, 0, s>>>(d_feats, T, stride, h->D, rows, gc, po, h->P, pdfs_per_cta, \
                                                      d_ll, ll_stride, bad)
  switch (h->DP / 4) {
    case 4: VB_LAUNCH(4); break;
    case 6: VB_LAUNCH(6); break;
    case 8: VB_LAUNCH(8); break;
    case 10: VB_LAUNCH(10); break;
    case 12: VB_LAUNCH(12); break;
    case 16: VB_LAUNCH(16); break;
    default: return fail(VBGPU_ERR_INVALID, "feature dim %d unsupported by the SIMT scorer (padded %d)", h->D, h->DP);
  }
#undef VB_LAUNCH
  VB_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace vb
