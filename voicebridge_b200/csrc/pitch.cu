// pitch.cu — Kaldi pitch extraction (ComputeKaldiPitch + ProcessPitch) for a batch of utterances on one B200.
//
// Replaces, behind vbgpu_pitch_*, the offline path of kaldi-master/src/feat/pitch-functions.cc
// (ComputeKaldiPitch :1291-1325 = OnlinePitchFeatureImpl::AcceptWaveform(whole wave) + InputFinished(), and
// ProcessPitch :1581-1595) and feat/resample.cc (LinearResample, ArbitraryResample).  frames_per_chunk = 0,
// simulate_first_pass_online = false, nccf_ballast_online = false, max_frames_latency = 0 (the defaults
// compute-kaldi-pitch-feats runs with).
//
// Data flow in HBM (one batch, utterances packed back to back):
//   wave (i16 / f32)  --k1 downsample-->  d_down [sum n2]   + per-utterance (sum, sumsq) of each call's samples
//   d_down            --k2 nccf------->   d_nccf [F][Sp] (ballasted NCCF on the log-spaced lag grid, the Viterbi input)
//                                         d_pov  [F][M]  (un-ballasted NCCF on the measured integer lags)
//   d_nccf            --k3 viterbi---->   d_bp [F][Sp] u16 back-pointers, then d_state[F] (one CTA per utterance)
//   d_state, d_pov    --k4 raw-------->   d_raw [F][2] = (NCCF at the chosen lag, pitch Hz), + POV / log-pitch side arrays
//   d_raw             --k5 process---->   out rows (pov feature, normalised log-pitch, delta-pitch, raw log-pitch)
// k1/k2/k4/k5 are embarrassingly parallel over samples / frames; k3 is sequential in time, parallel over lag states
// and utterances.  Every kernel is bound by instruction issue or latency, not HBM: the whole batch moves ~2 KB/frame.
#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "common.h"

using namespace vb;

namespace {

constexpr double k2Pi = 6.283185307179586476925286766559005;
constexpr double kPi = 3.1415926535897932384626433832795;

// LinearResample::FilterFunc / ArbitraryResample::FilterFunc (resample.cc:213-226, 318-331)
float filter_func(float t, float cutoff, int32_t num_zeros) {
  float window, filter;
  if (std::fabs(t) < num_zeros / (2.0 * cutoff)) window = (float)(0.5 * (1 + std::cos(k2Pi * cutoff / num_zeros * t)));
  else window = 0.0f;
  if (t != 0) filter = (float)(std::sin(k2Pi * cutoff * t) / (kPi * t));
  else filter = (float)(2 * cutoff);
  return filter * window;
}

int64_t gcd64(int64_t a, int64_t b) {
  while (b) {
    int64_t t = a % b;
    a = b;
    b = t;
  }
  return a;
}

struct UttDesc {          // one utterance of the batch
  int64_t in_off, n_in;   // samples in the packed input
  int64_t down_off;       // first down-sampled sample in d_down
  int64_t n1, n2;         // down-sampled samples after the first call / after the flush
  int64_t frame_off;      // first frame in the packed frame arrays
  int64_t row_off;        // first output row
  int32_t F1, F;          // frames produced by the first call / in total
  int32_t rows;           // output rows (F, or F + delay after ProcessPitch)
  int32_t pad;
};

struct PitchDev {  // plan tables on the device
  const int32_t *lr_first, *lr_nw;
  const float *lr_w;  // [out_unit][lr_max_w]
  int32_t in_unit, out_unit, lr_max_w;
  int64_t R;  // input samples the flush call still sees (LinearResample::SetRemainder)
  int32_t first_lag, M, S, Sp, W, shift, full, up_max;
  const int32_t *up_first, *up_n;
  const float *up_w;  // [up_max][S] (transposed: consecutive states are consecutive addresses)
  const float *soft_lag;  // soft_min_f0 * lags[i]
  const float *pitch_hz;  // 1 / lags[i]
  float preemph, nccf_ballast, factor;
  int32_t recompute_frame, snip_edges;
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- k1: LinearResample::Resample (resample.cc:120-160) for both calls, + the signal statistics --------------------
template <typename SampleT>
__global__ void __launch_bounds__(256) pitch_downsample_kernel(PitchDev p, const UttDesc *utts, const SampleT *wave,
                                                               float *down, double *stats) {
  const UttDesc u = utts[blockIdx.y];
  const SampleT *in = wave + u.in_off;
  double s0 = 0, q0 = 0, s1 = 0, q1 = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < u.n2; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t unit = i / p.out_unit;
    const int32_t ph = (int32_t)(i - unit * p.out_unit);
    const int64_t first = p.lr_first[ph] + unit * p.in_unit;
    const int32_t nw = p.lr_nw[ph];
    const float *w = p.lr_w + (size_t)ph * p.lr_max_w;
    const bool flush = i >= u.n1;  // second call: only the kept remainder of the input is visible
    const int64_t lo = flush ? max((int64_t)0, u.n_in - p.R) : 0;
    float acc = 0.f;
    for (int32_t k = 0; k < nw; k++) {
      const int64_t idx = first + k;
      if (idx >= lo && idx < u.n_in) acc = fmaf(w[k], (float)in[idx], acc);
    }
    down[u.down_off + i] = acc;
    if (flush) {
      s1 += acc;
      q1 += (double)acc * acc;
    } else {
      s0 += acc;
      q0 += (double)acc * acc;
    }
  }
  s0 = warp_sum_d(s0);
  q0 = warp_sum_d(q0);
  s1 = warp_sum_d(s1);
  q1 = warp_sum_d(q1);
  if ((threadIdx.x & 31) == 0) {
    double *st = stats + (size_t)blockIdx.y * 4;
    if (s0 != 0.0 || q0 != 0.0) {
      atomicAdd(st + 0, s0);
      atomicAdd(st + 1, q0);
    }
    if (s1 != 0.0 || q1 != 0.0) {
      atomicAdd(st + 2, s1);
      atomicAdd(st + 3, q1);
    }
  }
}

// ---- k1b: per-utterance energy terms (pitch-functions.cc:1110-1118, 949-992), once instead of per frame -------------
struct UttEnergy {
  float ballast[2];     // nccf_ballast_pitch of the first call's frames / of the flush call's frames
  float old_b, new_b;   // RecomputeBacktraces: ballast from the first call's energy / from the final energy
  int32_t rescale;      // 1 if the first call's frames are rescaled
  int32_t pad[3];
};

__device__ __forceinline__ bool approx_equal(float a, float b, float tol) {
  if (a == b) return true;
  const float diff = fabsf(a - b);
  if (isinf(diff) || diff != diff) return false;
  return diff <= tol * (fabsf(a) + fabsf(b));
}

__global__ void pitch_energy_kernel(PitchDev p, const UttDesc *utts, int32_t n_utts, const double *stats, UttEnergy *out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_utts) return;
  const UttDesc u = utts[k];
  const double *st = stats + (size_t)k * 4;
  // the reference adds float VecVec / Sum() results of each call to double totals
  const double sum1 = (double)(float)st[0], sq1 = (double)(float)st[1];
  const double sum2 = sum1 + (double)(float)st[2], sq2 = sq1 + (double)(float)st[3];
  const double ms1 = u.n1 > 0 ? sq1 / (double)u.n1 - (sum1 / (double)u.n1) * (sum1 / (double)u.n1) : 0.0;
  const double ms2 = u.n2 > 0 ? sq2 / (double)u.n2 - (sum2 / (double)u.n2) * (sum2 / (double)u.n2) : 0.0;
  UttEnergy e;
  e.ballast[0] = (float)((ms1 * p.W) * (ms1 * p.W) * (double)p.nccf_ballast);
  e.ballast[1] = (float)((ms2 * p.W) * (ms2 * p.W) * (double)p.nccf_ballast);
  e.old_b = e.new_b = 0.f;
  e.rescale = 0;
  e.pad[0] = e.pad[1] = e.pad[2] = 0;
  if (u.F1 > 0 && u.F1 < p.recompute_frame && u.n2 > 0) {
    const double mean2 = sum2 / (double)u.n2;
    const float ms_new = (float)(sq2 / (double)u.n2 - mean2 * mean2), ms_old = (float)ms1;
    if (!approx_equal(ms_old, ms_new, 0.01f)) {
      const float pw_new = ms_new * p.W, pw_old = ms_old * p.W;
      e.new_b = (float)((double)pw_new * (double)pw_new * (double)p.nccf_ballast);
      e.old_b = (float)((double)pw_old * (double)pw_old * (double)p.nccf_ballast);
      e.rescale = 1;
    }
  }
  out[k] = e;
}

// ---- k2: one warp per frame: ExtractFrame, ComputeCorrelation, ComputeNccf, ArbitraryResample, ballast rescale -------
// (pitch-functions.cc:839-901, 102-150, 1086-1135, 945-1002)
constexpr int kNccfWarps = 4;

__global__ void __launch_bounds__(kNccfWarps * 32) pitch_nccf_kernel(PitchDev p, const UttDesc *utts,
                                                                     const int32_t *frame2utt, int64_t frame_base,
                                                                     int64_t frame_end, const float *down,
                                                                     const UttEnergy *energy, float *nccf, float *pov) {
  extern __shared__ float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // two pad floats after the window (the sliding loads of the last lag overrun by two); up_max zero floats after m_pitch
  // (the up-sampling loop runs up_max taps for every state, the table is zero beyond a state's own taps)
  const int per_warp = p.full + 2 + 2 * p.M + p.up_max;
  float *win = smem + warp * per_warp, *m_pitch = win + p.full + 2, *m_pov = m_pitch + p.M + p.up_max;
  for (int i = lane; i < p.up_max; i += 32) m_pitch[p.M + i] = 0.f;
  const int64_t gf = frame_base + (int64_t)blockIdx.x * kNccfWarps + warp;
  if (gf >= frame_end) return;
  const int lo_u = frame2utt[gf];
  const UttDesc u = utts[lo_u];
  const int32_t f = (int32_t)(gf - u.frame_off);
  const bool call2 = f >= u.F1;
  const int64_t avail = call2 ? u.n2 : u.n1;
  const int64_t start = p.snip_edges ? (int64_t)f * p.shift : (int64_t)((f + 0.5) * p.shift) - p.full / 2;
  const int64_t vlo = start < 0 ? -start : 0, vhi = start + p.full > avail ? avail - start : p.full;
  const float *d = down + u.down_off + start;
  for (int i = lane; i < p.full + 2; i += 32) {
    float v = 0.f;
    if (i >= vlo && i < vhi) {
      v = d[i];
      if (p.preemph != 0.f) v = (i > vlo) ? __fsub_rn(v, __fmul_rn(p.preemph, d[i - 1])) : (float)((double)v * (1.0 - (double)p.preemph));
    }
    win[i] = v;
  }
  __syncwarp();
  const UttEnergy en = energy[lo_u];
  // zero-mean over the first W samples
  float s = 0.f;
  for (int i = lane; i < p.W; i += 32) s += win[i];
  const float mean = -warp_sum(s) / (float)p.W;
  for (int i = lane; i < p.full; i += 32) win[i] += mean;
  __syncwarp();
  float e1 = 0.f;
  for (int i = lane; i < p.W; i += 32) e1 = fmaf(win[i], win[i], e1);
  e1 = warp_sum(e1);
  const float ballast = en.ballast[call2 ? 1 : 0];
  float np_sum = 0.f;
  // Each lane owns three consecutive lags and slides a three-value register window over the signal: per sample one
  // broadcast load of win[i] and one stride-3 (conflict-free) load feed six FMAs.
  for (int base = 0; base < p.M; base += 96) {
    const int l0 = base + 3 * lane;
    if (l0 < p.M) {
      const float *w2 = win + p.first_lag + l0;
      float ip0 = 0.f, ip1 = 0.f, ip2 = 0.f, q0 = 0.f, q1 = 0.f, q2 = 0.f;
      float x0 = w2[0], x1 = w2[1];
#pragma unroll 6
      for (int i = 0; i < p.W; i++) {
        const float a = win[i], x2 = w2[i + 2];  // at most two floats past the window: the zero pad
        ip0 = fmaf(a, x0, ip0);
        ip1 = fmaf(a, x1, ip1);
        ip2 = fmaf(a, x2, ip2);
        q0 = fmaf(x0, x0, q0);
        q1 = fmaf(x1, x1, q1);
        q2 = fmaf(x2, x2, q2);
        x0 = x1;
        x1 = x2;
      }
#pragma unroll
      for (int k = 0; k < 3; k++) {
        const int l = l0 + k;
        if (l >= p.M) break;
        const float ip = k == 0 ? ip0 : (k == 1 ? ip1 : ip2), e2 = k == 0 ? q0 : (k == 1 ? q1 : q2);
        const float norm_prod = __fmul_rn(e1, e2);
        np_sum += norm_prod;
        float den = __fsqrt_rn(__fadd_rn(norm_prod, ballast));
        m_pitch[l] = den != 0.f ? __fdiv_rn(ip, den) : 0.f;
        den = __fsqrt_rn(norm_prod);
        const float pv = den != 0.f ? __fdiv_rn(ip, den) : 0.f;
        m_pov[l] = pv;
        pov[gf * p.M + l] = pv;
      }
    }
  }
  const float avg_norm = (float)((double)warp_sum(np_sum) / p.M);
  __syncwarp();
  // RecomputeBacktraces: frames of the first call are rescaled when the final energy estimate moved by more than 1%
  float scale = 1.f;
  if (en.rescale && !call2 && f < p.recompute_frame)
    scale = __fsqrt_rn(__fdiv_rn(__fadd_rn(en.old_b, avg_norm), __fadd_rn(en.new_b, avg_norm)));
  float *out = nccf + gf * p.Sp;
  for (int i = lane; i < p.Sp; i += 32) {
    float a = 0.f;
    if (i < p.S) {
      const float *m = m_pitch + p.up_first[i];
      const float *w = p.up_w + i;
#pragma unroll 4
      for (int j = 0; j < p.up_max; j++) a = fmaf(w[j * p.S], m[j], a);
      a = __fmul_rn(a, scale);
    }
    out[i] = a;
  }
}

// ---- k3: Viterbi over the lag states, one CTA per utterance (PitchFrameInfo::ComputeBacktraces :306-473;
// ComputeLocalCost :178-188; forward-cost renormalisation :1174-1176; SetBestState :486-512) ------------------------
// For state i the transition picks  argmin_j  fl(fl((j-i)^2) * factor) + prev[j]  (first minimum), evaluated with the
// reference's own FP32 expression.  The argmin is non-decreasing in i (the cost is a convex function of j - i plus a
// function of j) — the property the reference's interval-tightening search (:349-470) rests on.  Three levels:
//   (0) every 64th state ("anchor") scans all S predecessors, one warp per anchor;
//   (1) every 8th state scans [argmin(level-0 anchor below), argmin(level-0 anchor above)], eight lanes per state;
//   (2) every state scans the range between its two level-1 anchors.
// ~S/32 + 2 * 16 cost evaluations per thread and frame instead of S.
constexpr int kStride0 = 64, kStride1 = 8;

__device__ __forceinline__ float trans_cost(float df, float factor, float prev) {
  return __fadd_rn(__fmul_rn(__fmul_rn(df, df), factor), prev);  // (j - i) * (j - i) * inter_frame_factor + prev[j]
}

// G lanes (r = 0..G-1, consecutive lanes of one warp) find the first minimum over j in [lo, hi] for state a.
template <int G>
__device__ __forceinline__ void coop_scan(const float *fwd, float factor, int a, int lo, int hi, int r, float &best,
                                          int &bj) {
  const int len = hi - lo + 1, part = (len + G - 1) / G;
  const int j0 = lo + r * part, j1 = min(hi + 1, j0 + part);
  best = INFINITY;
  bj = max(0, min(j0, hi));
  float df = (float)(j0 - a);
#pragma unroll 4
  for (int j = j0; j < j1; j++) {
    const float cst = trans_cost(df, factor, fwd[j]);
    if (cst < best) {
      best = cst;
      bj = j;
    }
    df += 1.f;
  }
#pragma unroll
  for (int o = 1; o < G; o <<= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
    if (ob < best || (ob == best && oj < bj)) {
      best = ob;
      bj = oj;
    }
  }
}

// K lag states per thread (state i = tid + k * blockDim.x): the per-thread fixed work of a frame (barriers, reductions,
// range set-up) is paid once for K states, and an utterance needs only S / K threads.
constexpr int kLanes0 = 16, kLanes1 = 4;

template <int K>
__global__ void __launch_bounds__(K == 1 ? 1024 : (K == 2 ? 512 : 256)) pitch_viterbi_kernel(PitchDev p, const UttDesc *utts, const float *nccf,
                                                            uint16_t *bp, int32_t *state) {
  extern __shared__ float smem[];
  const int S = p.S;
  const int C0 = (S - 1 + kStride0 - 1) / kStride0;  // level-0 anchors 0..C0 at states min(64c, S-1)
  const int C1 = (S - 1 + kStride1 - 1) / kStride1;  // level-1 anchors 0..C1 at states min(8c, S-1)
  float *fwd = smem;                                 // [Sp] previous forward cost
  float *red = fwd + p.Sp;                           // [32]
  float *best1 = red + 32;                           // [C1+1]
  int *j1v = reinterpret_cast<int *>(best1 + C1 + 1);  // [C1+1]
  float *best0 = reinterpret_cast<float *>(j1v + C1 + 1);  // [C0+1]
  int *j0v = reinterpret_cast<int *>(best0 + C0 + 1);      // [C0+1]
  const UttDesc u = utts[blockIdx.x];
  if (u.F == 0) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthr = blockDim.x, nwarps = nthr >> 5;
  const int work0 = kLanes0 * (C0 + 1), iters0 = (work0 + nthr - 1) / nthr;
  const int work1 = kLanes1 * (C1 + 1), iters1 = (work1 + nthr - 1) / nthr;
  for (int k = tid; k < p.Sp; k += nthr) fwd[k] = 0.f;
  __syncthreads();
  const float factor = p.factor;
  const float *nc_row = nccf + u.frame_off * p.Sp;
  uint16_t *bp_row = bp + u.frame_off * p.Sp;
  float soft_lag[K], nc[K];
#pragma unroll
  for (int k = 0; k < K; k++) {
    const int i = tid + k * nthr;
    soft_lag[k] = i < S ? p.soft_lag[i] : 0.f;
    nc[k] = i < S ? nc_row[i] : 0.f;
  }
  for (int32_t f = 0; f < u.F; f++) {
    float nc_next[K];
#pragma unroll
    for (int k = 0; k < K; k++) {
      const int i = tid + k * nthr;
      nc_next[k] = (i < S && f + 1 < u.F) ? nc_row[(size_t)(f + 1) * p.Sp + i] : 0.f;
    }
    // level 0
    for (int it = 0; it < iters0; it++) {
      const int w = it * nthr + tid, c = w / kLanes0, r = w % kLanes0;
      const bool on = w < work0;
      float best;
      int bj;
      coop_scan<kLanes0>(fwd, factor, min(kStride0 * c, S - 1), 0, on ? S - 1 : -1, r, best, bj);
      if (on && r == 0) {
        best0[c] = best;
        j0v[c] = bj;
      }
    }
    __syncthreads();
    // level 1
    for (int it = 0; it < iters1; it++) {
      const int w = it * nthr + tid, c = w / kLanes1, r = w % kLanes1;
      const bool on = w < work1;
      const int a = min(kStride1 * c, S - 1);
      const bool is0 = on && (a == S - 1 || a % kStride0 == 0);  // also a level-0 anchor: copy
      const int c0 = a == S - 1 ? C0 : a / kStride0;
      int lo = 0, hi = -1;
      if (on && !is0) {
        lo = j0v[c0];
        hi = j0v[c0 + 1];
        if (lo > hi) {  // only when FP32 rounding breaks a tie the other way round
          const int t = lo;
          lo = hi;
          hi = t;
        }
      }
      float best;
      int bj;
      coop_scan<kLanes1>(fwd, factor, a, lo, hi, r, best, bj);
      if (on && r == 0) {
        best1[c] = is0 ? best0[c0] : best;
        j1v[c] = is0 ? j0v[c0] : bj;
      }
    }
    __syncthreads();
    // level 2 and the local cost, K states per thread
    float nxt[K], mn = INFINITY;
#pragma unroll
    for (int k = 0; k < K; k++) {
      const int i = tid + k * nthr;
      nxt[k] = INFINITY;
      if (i < S) {
        float best;
        int bj;
        if (i == S - 1 || i % kStride1 == 0) {
          const int ci = i == S - 1 ? C1 : i / kStride1;
          best = best1[ci];
          bj = j1v[ci];
        } else {
          const int c = i / kStride1;
          int lo = j1v[c], hi = j1v[c + 1];
          if (lo > hi) {
            const int t = lo;
            lo = hi;
            hi = t;
          }
          coop_scan<1>(fwd, factor, i, lo, hi, 0, best, bj);
        }
        float local = __fadd_rn(1.0f, -nc[k]);
        local = __fadd_rn(__fmul_rn(soft_lag[k], nc[k]), local);
        nxt[k] = __fadd_rn(best, local);
        bp_row[(size_t)f * p.Sp + i] = (uint16_t)bj;
        mn = fminf(mn, nxt[k]);
      }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    if (lane == 0) red[warp] = mn;
    __syncthreads();  // all reads of fwd / anchors are done, red is complete
    mn = red[lane < nwarps ? lane : 0];
#pragma unroll
    for (int o = 16; o; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
#pragma unroll
    for (int k = 0; k < K; k++) {
      const int i = tid + k * nthr;
      if (i < S) fwd[i] = __fsub_rn(nxt[k], mn);
      nc[k] = nc_next[k];
    }
    __syncthreads();
  }
  if (tid == 0) {
    int best = 0;
    for (int k = 1; k < S; k++)
      if (fwd[k] < fwd[best]) best = k;
    int32_t *st = state + u.frame_off;
    for (int32_t f = u.F - 1; f >= 0; f--) {
      st[f] = best;
      best = bp_row[(size_t)f * p.Sp + best];
    }
  }
}

// ---- k4: (NCCF at the chosen lag, pitch) per frame; POV and log-pitch for ProcessPitch -----------------------------
__device__ __forceinline__ float nccf_to_pov(float n) {  // pitch-functions.cc:78-87
  float ndash = fabsf(n);
  if (ndash > 1.0f) ndash = 1.0f;
  const float r = (float)(-5.2 + 5.4 * exp(7.5 * (ndash - 1.0)) + 4.8 * ndash - 2.0 * exp(-10.0 * ndash) +
                          4.2 * exp(20.0 * (ndash - 1.0)));
  return (float)(1.0 / (1 + exp(-1.0 * r)));
}
__device__ __forceinline__ float nccf_to_pov_feature(float n) {  // pitch-functions.cc:44-53
  n = fminf(1.0f, fmaxf(-1.0f, n));
  return (float)(pow(1.0001 - (double)n, 0.15) - 1.0);
}

__global__ void __launch_bounds__(256) pitch_raw_kernel(PitchDev p, int64_t total_frames, const int32_t *state,
                                                        const float *pov, float *raw, float *aux) {
  const int64_t gf = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gf >= total_frames) return;
  const int st = state[gf];
  const float *m = pov + gf * p.M + p.up_first[st];
  const int n = p.up_n[st];
  float a = 0.f;
  for (int j = 0; j < n; j++) a = fmaf(p.up_w[(size_t)j * p.S + st], m[j], a);
  const float hz = p.pitch_hz[st];
  raw[gf * 2] = a;
  raw[gf * 2 + 1] = hz;
  if (aux) {
    aux[gf * 2] = nccf_to_pov(a);
    aux[gf * 2 + 1] = logf(hz);
  }
}

// Host-supplied raw (NCCF, pitch) rows -> side arrays (vbgpu_pitch_process)
__global__ void __launch_bounds__(256) pitch_aux_kernel(int64_t total_frames, const float *raw, float *aux) {
  const int64_t gf = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gf >= total_frames) return;
  aux[gf * 2] = nccf_to_pov(raw[gf * 2]);
  aux[gf * 2 + 1] = logf(raw[gf * 2 + 1]);
}

// ---- k5: ProcessPitch (pitch-functions.cc:1414-1567), one thread per output row ------------------------------------
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16;
  x *= 0x7feb352du;
  x ^= x >> 15;
  x *= 0x846ca68bu;
  x ^= x >> 16;
  return x;
}

__global__ void __launch_bounds__(128) pitch_process_kernel(vbgpu_process_pitch_opts o, const UttDesc *utts,
                                                            int32_t n_utts, int64_t total_rows, const float *raw,
                                                            const float *aux, float *out, int32_t out_stride,
                                                            uint32_t seed) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= total_rows) return;
  int lo_u = 0, hi_u = n_utts - 1;
  while (lo_u < hi_u) {
    const int mid = (lo_u + hi_u + 1) >> 1;
    if (utts[mid].row_off <= row) lo_u = mid;
    else hi_u = mid - 1;
  }
  const UttDesc u = utts[lo_u];
  const int32_t t = (int32_t)(row - u.row_off), T = u.F;
  const int32_t f = t < o.delay ? 0 : t - o.delay;
  const float *r = raw + u.frame_off * 2, *a = aux + u.frame_off * 2;
  float *dst = out + row * out_stride;
  int idx = 0;
  const float log_pitch = a[f * 2 + 1];
  if (o.add_pov_feature) dst[idx++] = o.pov_scale * nccf_to_pov_feature(r[f * 2]) + o.pov_offset;
  if (o.add_normalized_log_pitch) {
    const int32_t b = max(0, f - o.normalization_left_context), e = min(T, f + o.normalization_right_context + 1);
    double sp = 0, slp = 0;
    for (int32_t g = b; g < e; g++) {
      const float pv = a[g * 2];
      sp += pv;
      slp += __fmul_rn(pv, a[g * 2 + 1]);
    }
    const float avg = (float)(slp / sp);
    dst[idx++] = (log_pitch - avg) * o.pitch_scale;
  }
  if (o.add_delta_pitch) {
    const int32_t w = o.delta_window;
    float norm = 0.f;
    for (int32_t k = -w; k <= w; k++) norm += (float)(k * k);
    const float inv_norm = (float)(1.0 / norm);
    float dlt = 0.f;
    for (int32_t k = -w; k <= w; k++) {
      if (k == 0) continue;
      const int32_t g = min(T - 1, max(0, f + k));
      dlt = __fadd_rn(dlt, __fmul_rn((float)k * inv_norm, a[g * 2 + 1]));
    }
    float noise = 0.f;
    if (o.delta_pitch_noise_stddev != 0.f) {  // RandGauss() * stddev, one draw per source frame; counter-based
      const uint32_t h1 = mix32(seed ^ mix32((uint32_t)(u.frame_off + f) * 2u + 1u));
      const uint32_t h2 = mix32(h1 ^ 0x9E3779B9u ^ (uint32_t)((u.frame_off + f) >> 31));
      const float u1 = ((h1 >> 8) + 1) * (1.0f / 16777217.0f), u2 = (h2 >> 8) * (1.0f / 16777216.0f);
      noise = sqrtf(-2.0f * logf(u1)) * cosf(6.2831853f * u2) * o.delta_pitch_noise_stddev;
    }
    dst[idx++] = (dlt + noise) * o.delta_pitch_scale;
  }
  if (o.add_raw_log_pitch) dst[idx++] = log_pitch;
}

}  // namespace

// ---- handle ---------------------------------------------------------------------------------------------------
struct vbgpu_pitch_s {
  vbgpu_pitch_opts o;
  int device = 0;
  vb::Stream stream, copy_stream;
  vb::Event ev_copied[4];
  int32_t in_hz = 0, out_hz = 0;
  int32_t last_lag = 0;
  PitchDev dev;
  DevBuf d_lr_first, d_lr_nw, d_lr_w, d_up_first, d_up_n, d_up_w, d_soft_lag, d_pitch_hz;
  DevBuf d_wave, d_down, d_stats, d_utts, d_nccf, d_pov, d_bp, d_state, d_raw, d_aux, d_out;
  DevBuf d_energy, d_frame_offsets, d_frame2utt;
  std::vector<UttDesc> utts;
  std::vector<int64_t> frame_offsets;
  uint32_t seed = 0x1234567u;
};

namespace {

int64_t num_out_samples(const vbgpu_pitch_s *h, int64_t n_in, bool flush) {  // resample.cc:57-80
  const int64_t tick_freq = (int64_t)h->in_hz / gcd64(h->in_hz, h->out_hz) * h->out_hz;
  const int64_t ticks_per_in = tick_freq / h->in_hz;
  int64_t len = n_in * ticks_per_in;
  if (!flush) {
    const float window_width = (float)(h->o.lowpass_filter_width / (2.0 * h->o.lowpass_cutoff));
    len -= (int32_t)std::floor(window_width * (int32_t)tick_freq);
  }
  if (len <= 0) return 0;
  const int64_t ticks_per_out = tick_freq / h->out_hz;
  int64_t last = len / ticks_per_out;
  if (last * ticks_per_out == len) last--;
  return last + 1;
}

int32_t frames_available(const vbgpu_pitch_s *h, int64_t n_down, bool finished) {  // pitch-functions.cc:768-792
  int32_t frame_length = h->dev.W;
  if (!finished) frame_length += h->last_lag;
  if (n_down < frame_length) return 0;
  if (!h->o.snip_edges) {
    if (finished) return (int32_t)(n_down * 1.0f / h->dev.shift + 0.5f);
    return (int32_t)((n_down - frame_length / 2) * 1.0f / h->dev.shift + 0.5f);
  }
  return (int32_t)((n_down - frame_length) / h->dev.shift + 1);
}

template <typename T>
int upload(DevBuf *b, const std::vector<T> &v, cudaStream_t s) {
  VB_TRY(b->reserve(std::max<size_t>(v.size(), 1) * sizeof(T)));
  if (!v.empty()) VB_CUDA(cudaMemcpyAsync(b->p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, s));
  return 0;
}

int build_plan(vbgpu_pitch_s *h) {  // OnlinePitchFeatureImpl ctor (pitch-functions.cc:715-766), resample.cc:34-106, 229-309
  const vbgpu_pitch_opts &o = h->o;
  PitchDev &d = h->dev;
  h->in_hz = (int32_t)o.samp_freq;
  h->out_hz = (int32_t)o.resample_freq;
  const int32_t base = (int32_t)gcd64(h->in_hz, h->out_hz);
  d.in_unit = h->in_hz / base;
  d.out_unit = h->out_hz / base;
  const double window_width = o.lowpass_filter_width / (2.0 * o.lowpass_cutoff);
  std::vector<int32_t> first(d.out_unit), nw(d.out_unit);
  d.lr_max_w = 0;
  for (int32_t i = 0; i < d.out_unit; i++) {
    const double output_t = i / (double)h->out_hz, min_t = output_t - window_width, max_t = output_t + window_width;
    const int32_t lo = (int32_t)std::ceil(min_t * h->in_hz), hi = (int32_t)std::floor(max_t * h->in_hz);
    first[i] = lo;
    nw[i] = hi - lo + 1;
    d.lr_max_w = std::max(d.lr_max_w, nw[i]);
  }
  std::vector<float> w((size_t)d.out_unit * d.lr_max_w, 0.f);
  for (int32_t i = 0; i < d.out_unit; i++) {
    const double output_t = i / (double)h->out_hz;
    for (int32_t j = 0; j < nw[i]; j++) {
      const double input_t = (first[i] + j) / (double)h->in_hz, delta_t = input_t - output_t;
      w[(size_t)i * d.lr_max_w + j] = filter_func((float)delta_t, o.lowpass_cutoff, o.lowpass_filter_width) / h->in_hz;
    }
  }
  d.R = (int64_t)std::ceil((float)(h->in_hz * o.lowpass_filter_width) / o.lowpass_cutoff);
  const double outer_min_lag = 1.0 / o.max_f0 - (o.upsample_filter_width / (2.0 * o.resample_freq));
  const double outer_max_lag = 1.0 / o.min_f0 + (o.upsample_filter_width / (2.0 * o.resample_freq));
  d.first_lag = (int32_t)std::ceil(o.resample_freq * outer_min_lag);
  h->last_lag = (int32_t)std::floor(o.resample_freq * outer_max_lag);
  d.M = h->last_lag + 1 - d.first_lag;
  d.W = (int32_t)(o.resample_freq * o.frame_length_ms / 1000.0);
  d.shift = (int32_t)(o.resample_freq * o.frame_shift_ms / 1000.0);
  d.full = d.W + h->last_lag;
  VB_CHECK(d.first_lag >= 0 && d.M > 0 && d.W > 0 && d.shift > 0, "pitch options give no lags / empty window");
  std::vector<float> lags;
  {
    const float min_lag = (float)(1.0 / o.max_f0), max_lag = (float)(1.0 / o.min_f0);
    for (float lag = min_lag; lag <= max_lag; lag = (float)(lag * (1.0 + o.delta_pitch))) {
      lags.push_back(lag);
      VB_CHECK(lags.size() <= 1024, "more than 1024 lag states (delta_pitch too small)");
    }
  }
  d.S = (int32_t)lags.size();
  d.Sp = (d.S + 31) / 32 * 32;
  VB_CHECK(d.S > 0, "no lag states");
  const float samp_rate_in = o.resample_freq, cutoff = (float)(o.resample_freq * 0.5);
  const int32_t nz = o.upsample_filter_width;
  const float off = -d.first_lag / o.resample_freq;
  const float filter_width = (float)(nz / (2.0 * cutoff));
  std::vector<int32_t> up_first(d.S), up_n(d.S);
  d.up_max = 0;
  for (int32_t i = 0; i < d.S; i++) {
    const float t = lags[i] + off, t_min = t - filter_width, t_max = t + filter_width;
    int32_t lo = (int32_t)std::ceil(samp_rate_in * t_min), hi = (int32_t)std::floor(samp_rate_in * t_max);
    lo = std::max(lo, 0);
    hi = std::min(hi, d.M - 1);
    up_first[i] = lo;
    up_n[i] = std::max(0, hi - lo + 1);
    d.up_max = std::max(d.up_max, up_n[i]);
  }
  std::vector<float> up_w((size_t)std::max(1, d.up_max) * d.S, 0.f), soft_lag(d.S), pitch_hz(d.S);
  for (int32_t i = 0; i < d.S; i++) {
    const float t = lags[i] + off;
    for (int32_t j = 0; j < up_n[i]; j++) {
      const float delta_t = t - (up_first[i] + j) / samp_rate_in;
      up_w[(size_t)j * d.S + i] = filter_func(delta_t, cutoff, nz) / samp_rate_in;
    }
    soft_lag[i] = o.soft_min_f0 * lags[i];
    pitch_hz[i] = (float)(1.0 / lags[i]);
  }
  const float delta_pitch_sq = (float)std::pow(std::log(1.0 + o.delta_pitch), 2.0);
  d.factor = delta_pitch_sq * o.penalty_factor;
  d.preemph = o.preemph_coeff;
  d.nccf_ballast = o.nccf_ballast;
  d.recompute_frame = o.recompute_frame;
  d.snip_edges = o.snip_edges;
  cudaStream_t s = h->stream;
  VB_TRY(upload(&h->d_lr_first, first, s));
  VB_TRY(upload(&h->d_lr_nw, nw, s));
  VB_TRY(upload(&h->d_lr_w, w, s));
  VB_TRY(upload(&h->d_up_first, up_first, s));
  VB_TRY(upload(&h->d_up_n, up_n, s));
  VB_TRY(upload(&h->d_up_w, up_w, s));
  VB_TRY(upload(&h->d_soft_lag, soft_lag, s));
  VB_TRY(upload(&h->d_pitch_hz, pitch_hz, s));
  VB_CUDA(cudaStreamSynchronize(s));
  d.lr_first = h->d_lr_first.as<int32_t>();
  d.lr_nw = h->d_lr_nw.as<int32_t>();
  d.lr_w = h->d_lr_w.as<float>();
  d.up_first = h->d_up_first.as<int32_t>();
  d.up_n = h->d_up_n.as<int32_t>();
  d.up_w = h->d_up_w.as<float>();
  d.soft_lag = h->d_soft_lag.as<float>();
  d.pitch_hz = h->d_pitch_hz.as<float>();
  return 0;
}

int process_dim(const vbgpu_process_pitch_opts *o) {
  return (o->add_pov_feature ? 1 : 0) + (o->add_normalized_log_pitch ? 1 : 0) + (o->add_delta_pitch ? 1 : 0) +
         (o->add_raw_log_pitch ? 1 : 0);
}

int check_process(const vbgpu_process_pitch_opts *o, int32_t out_stride) {
  VB_CHECK(process_dim(o) > 0, "ProcessPitch: at least one output feature must be selected (pitch-functions.cc:1407)");
  VB_CHECK(o->delay >= 0 && o->delta_window >= 1 && o->normalization_left_context >= 0 &&
               o->normalization_right_context >= 0,
           "bad ProcessPitch options");
  VB_CHECK(out_stride >= process_dim(o), "out_stride %d < %d output columns", out_stride, process_dim(o));
  return 0;
}

// Lay the batch out; returns total rows.
int plan_batch(vbgpu_pitch_s *h, const int64_t *sample_offsets, int32_t n_utts, const vbgpu_process_pitch_opts *proc,
               int64_t *total_down, int64_t *total_frames, int64_t *total_rows) {
  h->utts.resize(n_utts);
  int64_t down = 0, frames = 0, rows = 0;
  for (int32_t u = 0; u < n_utts; u++) {
    UttDesc &d = h->utts[u];
    d.in_off = sample_offsets[u];
    d.n_in = sample_offsets[u + 1] - sample_offsets[u];
    VB_CHECK(d.n_in >= 0, "sample_offsets not non-decreasing at utterance %d", u);
    d.n1 = num_out_samples(h, d.n_in, false);
    d.n2 = num_out_samples(h, d.n_in, true);
    d.F1 = frames_available(h, d.n1, false);
    d.F = frames_available(h, d.n2, true);
    d.F1 = std::min(d.F1, d.F);
    d.down_off = down;
    d.frame_off = frames;
    d.row_off = rows;
    d.rows = d.F > 0 ? d.F + (proc ? proc->delay : 0) : 0;
    d.pad = 0;
    down += (d.n2 + 3) / 4 * 4;
    frames += d.F;
    rows += d.rows;
  }
  *total_down = down;
  *total_frames = frames;
  *total_rows = rows;
  return 0;
}

template <typename SampleT>
int compute_impl(vbgpu_pitch_s *h, const SampleT *wave, const int64_t *sample_offsets, int32_t n_utts,
                 const vbgpu_process_pitch_opts *proc, float *out, int32_t out_stride) {
  VB_CHECK(h && sample_offsets && n_utts >= 0, "bad argument");
  if (n_utts == 0) return 0;
  VB_CHECK(sample_offsets[0] == 0, "sample_offsets[0] must be 0");
  if (proc) VB_TRY(check_process(proc, out_stride));
  else VB_CHECK(out_stride >= 2, "out_stride %d < 2", out_stride);
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  const PitchDev &p = h->dev;
  int64_t total_down, total_frames, total_rows;
  VB_TRY(plan_batch(h, sample_offsets, n_utts, proc, &total_down, &total_frames, &total_rows));
  if (total_frames == 0) return 0;
  VB_CHECK(wave && out, "null wave / out");
  const int64_t ns = sample_offsets[n_utts];
  VB_TRY(h->d_wave.reserve((size_t)ns * sizeof(SampleT)));
  VB_TRY(upload(&h->d_utts, h->utts, s));
  VB_TRY(h->d_down.reserve((size_t)total_down * 4));
  VB_TRY(h->d_stats.reserve((size_t)n_utts * 4 * 8));
  VB_TRY(h->d_nccf.reserve((size_t)total_frames * p.Sp * 4));
  VB_TRY(h->d_pov.reserve((size_t)total_frames * p.M * 4));
  VB_TRY(h->d_bp.reserve((size_t)total_frames * p.Sp * 2));
  VB_TRY(h->d_state.reserve((size_t)total_frames * 4));
  VB_TRY(h->d_raw.reserve((size_t)total_frames * 2 * 4));
  VB_TRY(h->d_aux.reserve((size_t)total_frames * 2 * 4));
  VB_CUDA(cudaMemsetAsync(h->d_stats.p, 0, (size_t)n_utts * 4 * 8, s));
  VB_TRY(h->d_energy.reserve((size_t)n_utts * sizeof(UttEnergy)));
  {  // frame -> utterance map
    h->frame_offsets.resize((size_t)n_utts + 1);
    for (int32_t k = 0; k < n_utts; k++) h->frame_offsets[k] = h->utts[k].frame_off;
    h->frame_offsets[n_utts] = total_frames;
    VB_TRY(upload(&h->d_frame_offsets, h->frame_offsets, s));
    VB_TRY(h->d_frame2utt.reserve((size_t)total_frames * 4));
    launch_fill_frame2utt(h->d_frame_offsets.as<int64_t>(), n_utts, total_frames, h->d_frame2utt.as<int32_t>(), s);
  }
  const UttDesc *d_utts = h->d_utts.as<UttDesc>();
  {
    // The PCM goes up in up to four groups of whole utterances on the copy stream; down-sampling, energy terms and the NCCF
    // of a group run while the next group is still crossing PCIe.  The Viterbi stays one launch over the whole batch (it
    // needs many utterances in flight: 7.8 ms for 256 utterances, 14.4 ms for 1 024).
    int n_groups = (int)std::min<int64_t>(4, std::max<int64_t>(1, (int64_t)ns * (int64_t)sizeof(SampleT) / (32ll << 20)));
    if (const char *e = std::getenv("VBGPU_PITCH_UPLOAD_GROUPS")) n_groups = std::max(1, std::min(4, std::atoi(e)));
    n_groups = std::min<int>(n_groups, n_utts);
    const size_t smem = (size_t)kNccfWarps * (p.full + 2 + 2 * p.M + p.up_max) * 4;
    VB_CHECK(smem <= 200 * 1024, "pitch window too long for shared memory (%zu bytes)", smem);
    if (smem > 48 * 1024)
      VB_CUDA(cudaFuncSetAttribute(pitch_nccf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VB_CUDA(cudaEventRecord(h->ev_copied[0], s));  // buffers of the previous call are free once stream s gets here
    VB_CUDA(cudaStreamWaitEvent(h->copy_stream, h->ev_copied[0], 0));
    int32_t u0 = 0;
    for (int g = 0; g < n_groups; g++) {
      int32_t u1 = u0;  // utterances [u0, u1): about ns / n_groups samples
      const int64_t want = g + 1 == n_groups ? ns : (ns * (g + 1)) / n_groups;
      while (u1 < n_utts && (g + 1 == n_groups || sample_offsets[u1 + 1] <= want || u1 == u0)) u1++;
      if (u1 == u0) continue;
      const int64_t s0 = sample_offsets[u0], s1 = sample_offsets[u1];
      if (s1 > s0)
        VB_CUDA(cudaMemcpyAsync(h->d_wave.as<SampleT>() + s0, wave + s0, (size_t)(s1 - s0) * sizeof(SampleT),
                                cudaMemcpyDefault, h->copy_stream));  // host or device PCM
      VB_CUDA(cudaEventRecord(h->ev_copied[g], h->copy_stream));
      VB_CUDA(cudaStreamWaitEvent(s, h->ev_copied[g], 0));
      const int32_t cnt = u1 - u0;
      int64_t max_n2 = 1;
      for (int32_t u = u0; u < u1; u++) max_n2 = std::max(max_n2, h->utts[u].n2);
      const int gx = (int)std::min<int64_t>((max_n2 + 255) / 256, 64);
      for (int32_t c0 = 0; c0 < cnt; c0 += 65535) {  // gridDim.y <= 65535
        const int32_t c = std::min<int32_t>(65535, cnt - c0);
        pitch_downsample_kernel<SampleT><<<dim3(gx, c), 256, 0, s>>>(p, d_utts + u0 + c0, h->d_wave.as<SampleT>(),
                                                                    h->d_down.as<float>(),
                                                                    h->d_stats.as<double>() + (size_t)(u0 + c0) * 4);
      }
      pitch_energy_kernel<<<(cnt + 127) / 128, 128, 0, s>>>(p, d_utts + u0, cnt, h->d_stats.as<double>() + (size_t)u0 * 4,
                                                           h->d_energy.as<UttEnergy>() + u0);
      const int64_t f0 = h->utts[u0].frame_off, f1 = u1 < n_utts ? h->utts[u1].frame_off : total_frames;
      if (f1 > f0) {
        const int64_t blocks = (f1 - f0 + kNccfWarps - 1) / kNccfWarps;
        pitch_nccf_kernel<<<(unsigned)blocks, kNccfWarps * 32, smem, s>>>(p, d_utts, h->d_frame2utt.as<int32_t>(), f0, f1,
                                                                         h->d_down.as<float>(), h->d_energy.as<UttEnergy>(),
                                                                         h->d_nccf.as<float>(), h->d_pov.as<float>());
      }
      VB_CUDA(cudaGetLastError());
      u0 = u1;
    }
  }
  {
    // Lag states per thread: small batches want many threads per utterance (latency), large ones few (instruction count).
    // Measured (256 / 512 / 1024 utterances): K=1 7.9 / 12.2 / 17.1 ms, K=2 7.8 / 10.6 / 14.8 ms, K=4 10.2 / 12.0 / 14.6 ms.
    int K = n_utts >= 8 * num_sms(h->device) ? 4 : (n_utts >= num_sms(h->device) ? 2 : 1);
    if (const char *e = std::getenv("VBGPU_PITCH_STATES_PER_THREAD")) K = std::atoi(e);  // measurement override
    const size_t smem = (size_t)(p.Sp + 32 + 2 * (p.S / kStride1 + 2) + 2 * (p.S / kStride0 + 2)) * 4;
    const int nthr = ((p.S + K - 1) / K + 31) / 32 * 32;
    if (K == 4)
      pitch_viterbi_kernel<4><<<n_utts, nthr, smem, s>>>(p, d_utts, h->d_nccf.as<float>(), h->d_bp.as<uint16_t>(),
                                                         h->d_state.as<int32_t>());
    else if (K == 2)
      pitch_viterbi_kernel<2><<<n_utts, nthr, smem, s>>>(p, d_utts, h->d_nccf.as<float>(), h->d_bp.as<uint16_t>(),
                                                         h->d_state.as<int32_t>());
    else
      pitch_viterbi_kernel<1><<<n_utts, ((p.S + 31) / 32) * 32, smem, s>>>(p, d_utts, h->d_nccf.as<float>(),
                                                                          h->d_bp.as<uint16_t>(), h->d_state.as<int32_t>());
  }
  pitch_raw_kernel<<<(unsigned)((total_frames + 255) / 256), 256, 0, s>>>(p, total_frames, h->d_state.as<int32_t>(),
                                                                         h->d_pov.as<float>(), h->d_raw.as<float>(),
                                                                         proc ? h->d_aux.as<float>() : nullptr);
  if (proc) {
    const int dim = process_dim(proc);
    VB_TRY(h->d_out.reserve((size_t)total_rows * dim * 4));
    pitch_process_kernel<<<(unsigned)((total_rows + 127) / 128), 128, 0, s>>>(*proc, d_utts, n_utts, total_rows,
                                                                             h->d_raw.as<float>(), h->d_aux.as<float>(),
                                                                             h->d_out.as<float>(), dim, h->seed++);
    VB_CUDA(cudaGetLastError());
    VB_CUDA(cudaMemcpy2DAsync(out, (size_t)out_stride * 4, h->d_out.p, (size_t)dim * 4, (size_t)dim * 4, total_rows,
                              cudaMemcpyDefault, s));
  } else {
    VB_CUDA(cudaGetLastError());
    VB_CUDA(cudaMemcpy2DAsync(out, (size_t)out_stride * 4, h->d_raw.p, 8, 8, total_frames, cudaMemcpyDefault, s));
  }
  VB_CUDA(cudaStreamSynchronize(s));
  return 0;
}

}  // namespace

extern "C" {

void vbgpu_pitch_opts_default(vbgpu_pitch_opts *o) {  // pitch-functions.h:103-123
  if (!o) return;
  *o = vbgpu_pitch_opts{16000.f, 10.f, 25.f, 0.f, 50.f, 400.f, 10.f, 0.1f, 1000.f, 4000.f, 0.005f, 7000.f, 1, 5, 500, 1};
}
void vbgpu_process_pitch_opts_default(vbgpu_process_pitch_opts *o) {  // pitch-functions.h:241-255
  if (!o) return;
  *o = vbgpu_process_pitch_opts{2.f, 2.f, 0.f, 10.f, 0.005f, 75, 75, 2, 0, 1, 1, 1, 0};
}

int vbgpu_pitch_create(const vbgpu_pitch_opts *opts, int device, vbgpu_pitch_t *out) {
  VB_CHECK(opts && out, "null argument");
  *out = nullptr;
  const vbgpu_pitch_opts &o = *opts;
  // LinearResample / ArbitraryResample constructor asserts (resample.cc:42-47, 236-240) and option sanity
  VB_CHECK(o.samp_freq > 0 && o.resample_freq > 0 && o.lowpass_cutoff > 0 && o.lowpass_filter_width > 0 &&
               o.upsample_filter_width > 0,
           "bad pitch resampling options");
  VB_CHECK(o.lowpass_cutoff * 2 <= o.samp_freq && o.lowpass_cutoff * 2 <= o.resample_freq,
           "lowpass_cutoff %g must be at most half of samp_freq %g and resample_freq %g", o.lowpass_cutoff, o.samp_freq,
           o.resample_freq);
  VB_CHECK(o.min_f0 > 0 && o.max_f0 > o.min_f0 && o.delta_pitch > 0 && o.frame_shift_ms > 0 && o.frame_length_ms > 0,
           "bad pitch search options");
  VB_TRY(vb::check_device(device));
  DeviceGuard g(device);
  std::unique_ptr<vbgpu_pitch_s, decltype(&vbgpu_pitch_destroy)> h(new vbgpu_pitch_s(), vbgpu_pitch_destroy);
  h->o = o;
  h->device = device;
  VB_TRY(h->stream.create());
  VB_TRY(h->copy_stream.create());
  for (vb::Event &ev : h->ev_copied) VB_TRY(ev.create());
  VB_TRY(build_plan(h.get()));
  *out = h.release();
  return 0;
}

void vbgpu_pitch_destroy(vbgpu_pitch_t h) {
  if (!h) return;
  DeviceGuard g(h->device);
  delete h;
}

int32_t vbgpu_pitch_num_states(vbgpu_pitch_t h) { return h ? h->dev.S : fail(VBGPU_ERR_INVALID, "null handle"); }

int64_t vbgpu_pitch_num_frames(vbgpu_pitch_t h, int64_t n_samples) {
  if (!h || n_samples < 0) return fail(VBGPU_ERR_INVALID, "bad argument");
  return frames_available(h, num_out_samples(h, n_samples, true), true);
}

int vbgpu_pitch_compute_f32(vbgpu_pitch_t h, const float *wave, const int64_t *sample_offsets, int32_t n_utts,
                            const vbgpu_process_pitch_opts *process, float *out, int32_t out_stride) {
  return compute_impl<float>(h, wave, sample_offsets, n_utts, process, out, out_stride);
}

int vbgpu_pitch_compute_i16(vbgpu_pitch_t h, const int16_t *pcm, const int64_t *sample_offsets, int32_t n_utts,
                            const vbgpu_process_pitch_opts *process, float *out, int32_t out_stride) {
  return compute_impl<int16_t>(h, pcm, sample_offsets, n_utts, process, out, out_stride);
}

int vbgpu_pitch_process(vbgpu_pitch_t h, const vbgpu_process_pitch_opts *process, const float *raw, int32_t raw_stride,
                        const int64_t *frame_offsets, int32_t n_utts, float *out, int32_t out_stride) {
  VB_CHECK(h && process && frame_offsets && n_utts >= 0 && raw_stride >= 2, "bad argument");
  VB_TRY(check_process(process, out_stride));
  if (n_utts == 0) return 0;
  VB_CHECK(frame_offsets[0] == 0, "frame_offsets[0] must be 0");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  h->utts.assign(n_utts, UttDesc());
  int64_t rows = 0;
  for (int32_t u = 0; u < n_utts; u++) {
    UttDesc &d = h->utts[u];
    const int64_t T = frame_offsets[u + 1] - frame_offsets[u];
    VB_CHECK(T >= 0 && T < (1ll << 31), "bad frame_offsets at utterance %d", u);
    d.frame_off = frame_offsets[u];
    d.F = d.F1 = (int32_t)T;
    d.row_off = rows;
    d.rows = T > 0 ? (int32_t)T + process->delay : 0;
    rows += d.rows;
  }
  const int64_t total_frames = frame_offsets[n_utts];
  if (total_frames == 0) return 0;
  VB_CHECK(raw && out, "null raw / out");
  for (int64_t t = 0; t < total_frames; t++)
    VB_CHECK(raw[t * raw_stride + 1] > 0, "pitch %g <= 0 at frame %lld (pitch-functions.cc:1472)",
             raw[t * raw_stride + 1], (long long)t);
  const int dim = process_dim(process);
  VB_TRY(upload(&h->d_utts, h->utts, s));
  VB_TRY(h->d_raw.reserve((size_t)total_frames * 8));
  VB_TRY(h->d_aux.reserve((size_t)total_frames * 8));
  VB_TRY(h->d_out.reserve((size_t)rows * dim * 4));
  VB_CUDA(cudaMemcpy2DAsync(h->d_raw.p, 8, raw, (size_t)raw_stride * 4, 8, total_frames, cudaMemcpyHostToDevice, s));
  pitch_aux_kernel<<<(unsigned)((total_frames + 255) / 256), 256, 0, s>>>(total_frames, h->d_raw.as<float>(),
                                                                         h->d_aux.as<float>());
  pitch_process_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, s>>>(*process, h->d_utts.as<UttDesc>(), n_utts, rows,
                                                                     h->d_raw.as<float>(), h->d_aux.as<float>(),
                                                                     h->d_out.as<float>(), dim, h->seed++);
  VB_CUDA(cudaGetLastError());
  VB_CUDA(cudaMemcpy2DAsync(out, (size_t)out_stride * 4, h->d_out.p, (size_t)dim * 4, (size_t)dim * 4, rows,
                            cudaMemcpyDeviceToHost, s));
  VB_CUDA(cudaStreamSynchronize(s));
  return 0;
}

}  // extern "C"
