// align.cu — forced alignment: the Viterbi search of gmm-align-compiled (AlignUtteranceWrapper -> FasterDecoder::Decode /
// GetBestPath) over each utterance's training graph, for a packed batch of whole utterances.  The search is exact (no
// beam).  Semantics, tie rule and limits are stated in include/vbgpu.h (vbgpu_align_*).
//
// Create time (host): every graph is checked, then laid out for the kernels —
//   * the incoming arcs of every state, emitting ones and epsilon ones in two CSR lists by destination, each arc stored
//     as {src, subset column, weight, original arc index} in original arc order (the tie rule);
//   * the epsilon levels: level(s) = the longest epsilon path into s (Kahn's topological sort, which also finds cycles);
//     the states of level >= 1 are listed level by level, so one barrier per level relaxes the epsilon closure exactly;
//   * the pdf subset of every utterance: the distinct tid2pdf of its emitting arcs in increasing order (what
//     vbgpu::PdfsOfGraph lists); an emitting arc's column is its pdf's position there.
// Call time: the subset log-likelihoods come from the model's subset scorer (capi.cu), then per group of utterances
//   align_viterbi_kernel    a CTA per utterance.  State costs in shared memory, FP64, double-buffered; the next frame's
//                           subset row is staged into shared memory (cp.async) while the current frame is relaxed.  Per
//                           frame: a thread per destination state scans its incoming emitting arcs with a strict <, then
//                           the epsilon levels, each behind a barrier.  One traceback entry (winning arc, -1 = none) per
//                           (frame, state) goes to global memory; the best cost + final is a block reduction.
//   align_traceback_kernel  a thread per utterance walks the entries back from the best final state (epsilon arcs
//                           included) and writes the transition-id and pdf-id of every frame.
#include <cuda_pipeline.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "common.h"

namespace {

// 256 threads per utterance (a few states each at the bench shape); __launch_bounds__(kThreads, 6) below holds the Viterbi
// kernel to 39 registers, six CTAs per SM, without spills (left alone, ptxas picks 32 registers and spills).
constexpr int kThreads = 256;

// shared memory of one CTA: 2 S doubles of costs + 2 n_sub floats of staged log-likelihood rows
size_t smem_bytes(int32_t S, int32_t n_sub) { return (size_t)S * 16 + (size_t)n_sub * 8; }

__device__ __forceinline__ void stage_row(float *dst, const float *src, int32_t n) {
  for (int j = threadIdx.x; j < n; j += kThreads) __pipeline_memcpy_async(dst + j, src + j, 4);
  __pipeline_commit();
}

// Epsilon closure of frame row c / tbr, level after level (level 0 states have no incoming epsilon arc).  An epsilon
// relaxation replaces a cost only if it is strictly lower; among the arcs into one state the first in arc order wins.
template <typename TB>
__device__ __forceinline__ void eps_closure(double *c, TB *tbr, const vb::AlignUtt &U, const int32_t *__restrict__ xo,
                                            const int4 *__restrict__ arcs, const int32_t *__restrict__ lvl_off,
                                            const int32_t *__restrict__ lvl_states) {
  for (int l = 0; l < U.n_lvls; l++) {
    __syncthreads();
    const int i1 = lvl_off[U.lvl_base + l + 1];
    for (int i = lvl_off[U.lvl_base + l] + threadIdx.x; i < i1; i += kThreads) {
      const int s = lvl_states[i];
      double best = c[s];
      int arg = -1;
      for (int a = xo[s]; a < xo[s + 1]; a++) {
        const int4 A = __ldg(arcs + a);
        const double v = c[A.x] + (double)__int_as_float(A.z);
        if (v < best) best = v, arg = A.w;
      }
      if (arg >= 0) c[s] = best, tbr[s] = (TB)arg;
    }
  }
}

template <typename TB>
__global__ void __launch_bounds__(kThreads, 6) align_viterbi_kernel(
    const vb::AlignUtt *__restrict__ utts, const vb::AlignCall *__restrict__ calls, int32_t u0,
    const int32_t *__restrict__ e_off, const int32_t *__restrict__ x_off, const int4 *__restrict__ arcs,
    const int32_t *__restrict__ lvl_off, const int32_t *__restrict__ lvl_states, const float *__restrict__ finals,
    const float *__restrict__ ll, float scale, TB *__restrict__ tb, double *__restrict__ tot_cost,
    int32_t *__restrict__ best_state) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ double red_c[kThreads / 32];
  __shared__ int red_s[kThreads / 32];
  const int u = u0 + blockIdx.x;
  const vb::AlignUtt U = utts[u];
  const vb::AlignCall C = calls[u];
  const int S = U.S, T = (int)C.T;
  double *const cost0 = reinterpret_cast<double *>(smem), *const cost1 = cost0 + S;
  float *const row0 = reinterpret_cast<float *>(cost1 + S), *const row1 = row0 + U.n_sub;
  const int32_t *eo = e_off + U.csr_base, *xo = x_off + U.csr_base;
  const float *llu = ll + C.ll_off;
  TB *tbu = tb + C.tb_off;
  const double kInf = __longlong_as_double(0x7ff0000000000000LL);

  for (int s = threadIdx.x; s < S; s += kThreads) {
    cost0[s] = s == U.start ? 0.0 : kInf;
    tbu[s] = (TB)-1;
  }
  if (T > 0) stage_row(row0, llu, U.n_sub);
  eps_closure(cost0, tbu, U, xo, arcs, lvl_off, lvl_states);  // (its first barrier orders the initialisation)
  for (int t = 0; t < T; t++) {
    __pipeline_wait_prior(0);
    __syncthreads();  // row t staged by every thread; the previous frame's closure complete
    const bool odd = t & 1;
    if (t + 1 < T) stage_row(odd ? row0 : row1, llu + (int64_t)(t + 1) * U.n_sub, U.n_sub);
    const double *prev = odd ? cost1 : cost0;
    double *cur = odd ? cost0 : cost1;
    const float *r = odd ? row1 : row0;
    TB *tbr = tbu + (int64_t)(t + 1) * S;
    for (int s = threadIdx.x; s < S; s += kThreads) {
      double best = kInf;
      int arg = -1;
      for (int a = eo[s]; a < eo[s + 1]; a++) {
        const int4 A = __ldg(arcs + a);
        const float ac = -__fmul_rn(scale, r[A.y]);
        const double v = (prev[A.x] + (double)__int_as_float(A.z)) + (double)ac;
        if (v < best) best = v, arg = A.w;
      }
      cur[s] = best;
      tbr[s] = (TB)arg;
    }
    eps_closure(cur, tbr, U, xo, arcs, lvl_off, lvl_states);
  }
  __syncthreads();

  // best of cost + final; equal costs go to the lower state
  const double *c = (T & 1) ? cost1 : cost0;
  double bc = kInf;
  int bs = -1;
  for (int s = threadIdx.x; s < S; s += kThreads) {
    const double v = c[s] + (double)finals[U.state_base + s];
    if (v < bc) bc = v, bs = s;
  }
  auto better = [](double oc, int os, double bc, int bs) {
    return os >= 0 && (bs < 0 || oc < bc || (oc == bc && os < bs));
  };
  for (int o = 16; o > 0; o >>= 1) {
    const double oc = __shfl_down_sync(0xffffffffu, bc, o);
    const int os = __shfl_down_sync(0xffffffffu, bs, o);
    if (better(oc, os, bc, bs)) bc = oc, bs = os;
  }
  if ((threadIdx.x & 31) == 0) red_c[threadIdx.x >> 5] = bc, red_s[threadIdx.x >> 5] = bs;
  __syncthreads();
  if (threadIdx.x == 0) {
    bc = red_c[0], bs = red_s[0];
    for (int w = 1; w < kThreads / 32; w++)
      if (better(red_c[w], red_s[w], bc, bs)) bc = red_c[w], bs = red_s[w];
    tot_cost[u] = bs >= 0 ? bc : kInf;
    best_state[u] = bs;
  }
}

// A thread per utterance: from the best final state at row T back to the start state at row 0.  An utterance without a
// reachable final state gets transition-id 0 and pdf-id -1 on every frame.
template <typename TB>
__global__ void __launch_bounds__(64) align_traceback_kernel(
    const vb::AlignUtt *__restrict__ utts, const vb::AlignCall *__restrict__ calls, int32_t u0, int32_t n,
    const TB *__restrict__ tb, const int32_t *__restrict__ a_src, const int32_t *__restrict__ a_lab,
    const int32_t *__restrict__ tid2pdf, const int32_t *__restrict__ best_state, int32_t *__restrict__ ali,
    int32_t *__restrict__ pdf_ids) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int u = u0 + i;
  const vb::AlignUtt U = utts[u];
  const vb::AlignCall C = calls[u];
  int32_t *al = ali + C.f0, *pd = pdf_ids ? pdf_ids + C.f0 : nullptr;
  int s = best_state[u];
  if (s < 0) {
    for (int64_t t = 0; t < C.T; t++) {
      al[t] = 0;
      if (pd) pd[t] = -1;
    }
    return;
  }
  const TB *tbu = tb + C.tb_off;
  int64_t r = C.T;
  for (;;) {
    const int a = (int)tbu[r * U.S + s];
    if (a < 0) break;
    const int lab = a_lab[U.arc_base + a];
    s = a_src[U.arc_base + a];
    if (lab) {
      --r;
      al[r] = lab;
      if (pd) pd[r] = tid2pdf[lab];
    }
  }
}

// The arcs' weights for this call: the graph's own, plus tid_cost[ilabel] (float, as fst::Times) on emitting arcs.
__global__ void align_weights_kernel(const float *__restrict__ base_w, const int32_t *__restrict__ lab,
                                     const float *__restrict__ tid_cost, int4 *__restrict__ arcs, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float w = base_w[i];
    reinterpret_cast<float *>(arcs + i)[2] = (tid_cost && lab[i]) ? __fadd_rn(w, tid_cost[lab[i]]) : w;
  }
}

bool bad_cost(float v) { return std::isnan(v) || v == -INFINITY; }

}  // namespace

namespace vb {

int align_create(int32_t n_utts, const int32_t *state_offsets, const int32_t *start, const float *final_cost,
                 const int64_t *arc_offsets, const int32_t *arc_src, const int32_t *arc_dst, const int32_t *arc_ilabel,
                 const float *arc_weight, const int32_t *tid2pdf, int32_t num_tids, int device, vbgpu_align_t *out) {
  VB_CHECK(out, "null argument");
  *out = nullptr;
  VB_CHECK(n_utts >= 1 && num_tids >= 0, "n_utts %d / num_tids %d out of range", n_utts, num_tids);
  VB_CHECK(state_offsets && start && final_cost && arc_offsets && tid2pdf, "null graph array");
  VB_CHECK(state_offsets[0] == 0 && arc_offsets[0] == 0, "state_offsets / arc_offsets must start at 0");
  for (int32_t u = 0; u < n_utts; u++) {
    const int64_t S = (int64_t)state_offsets[u + 1] - state_offsets[u], A = arc_offsets[u + 1] - arc_offsets[u];
    VB_CHECK(S >= 1, "utterance %d has no states", u);
    VB_CHECK(S <= kAlignMaxStates, "utterance %d has %lld states, more than the %d the alignment kernel supports", u,
             (long long)S, kAlignMaxStates);
    VB_CHECK(A >= 0, "arc_offsets decrease at utterance %d", u);
    VB_CHECK(start[u] >= 0 && start[u] < S, "utterance %d: start state %d outside [0, %lld)", u, start[u], (long long)S);
  }
  const int64_t n_states = state_offsets[n_utts], n_arcs = arc_offsets[n_utts];
  VB_CHECK(n_arcs < (1ll << 31) && n_states + n_utts < (1ll << 31), "too many arcs / states in one handle");
  VB_CHECK(n_arcs == 0 || (arc_src && arc_dst && arc_ilabel && arc_weight), "null arc array");
  int32_t max_pdf = -1;
  for (int32_t i = 1; i <= num_tids; i++) {
    VB_CHECK(tid2pdf[i] >= 0, "tid2pdf[%d] = %d is negative", i, tid2pdf[i]);
    max_pdf = std::max(max_pdf, tid2pdf[i]);
  }
  for (int64_t i = 0; i < n_states; i++) VB_CHECK(!bad_cost(final_cost[i]), "final cost of state %lld is NaN or -inf", (long long)i);

  std::vector<AlignUtt> utts((size_t)n_utts);
  std::vector<int32_t> e_off((size_t)(n_states + n_utts)), x_off((size_t)(n_states + n_utts));
  std::vector<int4> arcs((size_t)n_arcs);
  std::vector<float> cw((size_t)n_arcs);
  std::vector<int32_t> clab((size_t)n_arcs), lvl_off, lvl_states;
  std::vector<int64_t> sub_off((size_t)n_utts + 1, 0);
  std::vector<int32_t> sub_pdfs, h_S((size_t)n_utts), h_nsub((size_t)n_utts);
  bool wide = false;  // some utterance has 32768 arcs or more: int32 traceback entries
  std::vector<int32_t> cnt, level, indeg, queue, col_of;
  for (int32_t u = 0; u < n_utts; u++) {
    const int32_t S = state_offsets[u + 1] - state_offsets[u];
    const int64_t a0 = arc_offsets[u], a1 = arc_offsets[u + 1];
    const int32_t A = (int32_t)(a1 - a0);
    wide |= A >= 32768;
    for (int64_t a = a0; a < a1; a++) {
      VB_CHECK(arc_src[a] >= 0 && arc_src[a] < S && arc_dst[a] >= 0 && arc_dst[a] < S,
               "utterance %d, arc %lld: src %d / dst %d outside the utterance's %d states", u, (long long)(a - a0),
               arc_src[a], arc_dst[a], S);
      VB_CHECK(arc_ilabel[a] >= 0 && arc_ilabel[a] <= num_tids, "utterance %d, arc %lld: ilabel %d outside [0, %d]", u,
               (long long)(a - a0), arc_ilabel[a], num_tids);
      VB_CHECK(!bad_cost(arc_weight[a]), "utterance %d, arc %lld: weight is NaN or -inf", u, (long long)(a - a0));
    }
    // epsilon levels (Kahn): level(dst) = max over epsilon arcs of level(src) + 1
    level.assign((size_t)S, 0);
    indeg.assign((size_t)S, 0);
    cnt.assign((size_t)S + 1, 0);
    for (int64_t a = a0; a < a1; a++)
      if (arc_ilabel[a] == 0) indeg[arc_dst[a]]++, cnt[arc_src[a] + 1]++;
    for (int32_t s = 0; s < S; s++) cnt[s + 1] += cnt[s];
    std::vector<int32_t> out_eps((size_t)cnt[S]), fill(cnt.begin(), cnt.end() - 1);
    for (int64_t a = a0; a < a1; a++)
      if (arc_ilabel[a] == 0) out_eps[fill[arc_src[a]]++] = arc_dst[a];
    queue.clear();
    for (int32_t s = 0; s < S; s++)
      if (!indeg[s]) queue.push_back(s);
    for (size_t q = 0; q < queue.size(); q++) {
      const int32_t s = queue[q];
      for (int32_t k = cnt[s]; k < cnt[s + 1]; k++) {
        const int32_t d = out_eps[k];
        level[d] = std::max(level[d], level[s] + 1);
        if (--indeg[d] == 0) queue.push_back(d);
      }
    }
    VB_CHECK((int32_t)queue.size() == S, "utterance %d: its epsilon arcs form a cycle", u);
    const int32_t n_lvls = S ? *std::max_element(level.begin(), level.end()) : 0;
    AlignUtt &U = utts[u];
    U.S = S;
    U.start = start[u];
    U.n_lvls = n_lvls;
    U.state_base = state_offsets[u];
    U.csr_base = state_offsets[u] + u;
    U.lvl_base = (int32_t)lvl_off.size();
    U.arc_base = (int32_t)a0;
    for (int32_t l = 1; l <= n_lvls; l++) {
      lvl_off.push_back((int32_t)lvl_states.size());
      for (int32_t s = 0; s < S; s++)
        if (level[s] == l) lvl_states.push_back(s);
    }
    lvl_off.push_back((int32_t)lvl_states.size());
    // pdf subset, in increasing pdf order
    const size_t sub0 = sub_pdfs.size();
    for (int64_t a = a0; a < a1; a++)
      if (arc_ilabel[a]) sub_pdfs.push_back(tid2pdf[arc_ilabel[a]]);
    std::sort(sub_pdfs.begin() + sub0, sub_pdfs.end());
    sub_pdfs.erase(std::unique(sub_pdfs.begin() + sub0, sub_pdfs.end()), sub_pdfs.end());
    const int32_t n_sub = (int32_t)(sub_pdfs.size() - sub0);
    VB_CHECK(n_sub <= kAlignMaxSubset, "utterance %d reads %d distinct pdfs, more than the %d the alignment kernel stages",
             u, n_sub, kAlignMaxSubset);
    U.n_sub = n_sub;
    sub_off[u + 1] = sub_off[u] + n_sub;
    h_S[u] = S;
    h_nsub[u] = n_sub;
    // incoming arcs by destination, emitting ones first, each list in arc order
    int32_t *eo = e_off.data() + U.csr_base, *xo = x_off.data() + U.csr_base;
    std::fill(eo, eo + S + 1, 0);
    std::fill(xo, xo + S + 1, 0);
    for (int64_t a = a0; a < a1; a++) (arc_ilabel[a] ? eo : xo)[arc_dst[a] + 1]++;
    for (int32_t s = 0; s < S; s++) eo[s + 1] += eo[s];
    for (int32_t s = 0; s <= S; s++) xo[s] += eo[S];
    for (int32_t s = 0; s < S; s++) xo[s + 1] += xo[s] - eo[S];
    for (int32_t s = 0; s <= S; s++) eo[s] += (int32_t)a0, xo[s] += (int32_t)a0;
    std::vector<int32_t> put(eo, eo + S), putx(xo, xo + S);
    for (int64_t a = a0; a < a1; a++) {
      const int32_t lab = arc_ilabel[a], d = arc_dst[a];
      const int32_t k = lab ? put[d]++ : putx[d]++;
      const int32_t col = lab ? (int32_t)(std::lower_bound(sub_pdfs.begin() + sub0, sub_pdfs.end(), tid2pdf[lab]) -
                                          (sub_pdfs.begin() + sub0))
                              : -1;
      int32_t wbits;
      std::memcpy(&wbits, arc_weight + a, 4);
      arcs[k] = make_int4(arc_src[a], col, wbits, (int32_t)(a - a0));
      cw[k] = arc_weight[a];
      clab[k] = lab;
    }
  }

  VB_TRY(check_device(device));
  DeviceGuard g(device);
  std::unique_ptr<vbgpu_align_s, decltype(&vbgpu_align_destroy)> h(new vbgpu_align_s, vbgpu_align_destroy);
  h->device = device;
  h->n_utts = n_utts;
  h->num_tids = num_tids;
  h->n_arcs = n_arcs;
  h->max_pdf = max_pdf;
  h->tb_bytes = wide ? 4 : 2;
  h->h_S = std::move(h_S);
  h->h_nsub = std::move(h_nsub);
  h->h_sub_off = std::move(sub_off);
  h->h_sub_pdfs = std::move(sub_pdfs);
  if (h->h_sub_pdfs.empty()) h->h_sub_pdfs.push_back(0);  // (a valid pointer for the scorer when nothing emits)
  if (lvl_off.empty()) lvl_off.push_back(0);
  if (lvl_states.empty()) lvl_states.push_back(0);
  VB_TRY(h->stream.create());
  VB_TRY(h->d_utts.upload(utts.data(), utts.size() * sizeof(AlignUtt)));
  VB_TRY(h->d_eoff.upload(e_off.data(), e_off.size() * 4));
  VB_TRY(h->d_xoff.upload(x_off.data(), x_off.size() * 4));
  VB_TRY(h->d_lvl_off.upload(lvl_off.data(), lvl_off.size() * 4));
  VB_TRY(h->d_lvl_states.upload(lvl_states.data(), lvl_states.size() * 4));
  VB_TRY(h->d_final.upload(final_cost, (size_t)n_states * 4));
  VB_TRY(h->d_tid2pdf.upload(tid2pdf, (size_t)(num_tids + 1) * 4));
  if (n_arcs) {
    VB_TRY(h->d_arcs.upload(arcs.data(), arcs.size() * 16));
    VB_TRY(h->d_cw.upload(cw.data(), cw.size() * 4));
    VB_TRY(h->d_clab.upload(clab.data(), clab.size() * 4));
    VB_TRY(h->d_asrc.upload(arc_src, (size_t)n_arcs * 4));
    VB_TRY(h->d_alab.upload(arc_ilabel, (size_t)n_arcs * 4));
  }
  VB_TRY(h->d_best.reserve((size_t)n_utts * 4));
  VB_TRY(h->d_calls.reserve((size_t)n_utts * sizeof(AlignCall)));
  const int max_smem = (int)smem_bytes(kAlignMaxStates, kAlignMaxSubset);
  VB_CUDA(cudaFuncSetAttribute(align_viterbi_kernel<int16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
  VB_CUDA(cudaFuncSetAttribute(align_viterbi_kernel<int32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
  *out = h.release();
  return 0;
}

int align_set_weights(vbgpu_align_t h, const float *tid_cost, cudaStream_t s) {
  const int64_t n_arcs = h->n_arcs;
  if (n_arcs == 0) return 0;
  const float *d_tc = nullptr;
  if (tid_cost) {
    VB_TRY(h->d_tid_cost.reserve((size_t)(h->num_tids + 1) * 4));
    VB_CUDA(cudaMemcpyAsync(h->d_tid_cost.p, tid_cost, (size_t)(h->num_tids + 1) * 4, cudaMemcpyHostToDevice, s));
    d_tc = h->d_tid_cost.as<float>();
  }
  const int64_t blocks = std::min<int64_t>((n_arcs + 255) / 256, 148 * 8);
  align_weights_kernel<<<(unsigned)blocks, 256, 0, s>>>(h->d_cw.as<float>(), h->d_clab.as<int32_t>(), d_tc,
                                                        h->d_arcs.as<int4>(), n_arcs);
  VB_CUDA(cudaGetLastError());
  return 0;
}

int align_group_launch(vbgpu_align_t h, int32_t u0, int32_t n, int32_t max_S, int32_t max_sub, const float *d_ll,
                       float acoustic_scale, void *d_tb, int32_t *d_ali, int32_t *d_pdf_ids, double *d_tot_cost,
                       cudaStream_t s) {
  if (n == 0) return 0;
  const size_t smem = smem_bytes(max_S, max_sub);
  const AlignUtt *utts = h->d_utts.as<AlignUtt>();
  const AlignCall *calls = h->d_calls.as<AlignCall>();
  const int32_t *lab = h->d_alab.as<int32_t>(), *src = h->d_asrc.as<int32_t>();
  if (h->tb_bytes == 2) {
    align_viterbi_kernel<int16_t><<<n, kThreads, smem, s>>>(
        utts, calls, u0, h->d_eoff.as<int32_t>(), h->d_xoff.as<int32_t>(), h->d_arcs.as<int4>(), h->d_lvl_off.as<int32_t>(),
        h->d_lvl_states.as<int32_t>(), h->d_final.as<float>(), d_ll, acoustic_scale, static_cast<int16_t *>(d_tb),
        d_tot_cost, h->d_best.as<int32_t>());
    VB_CUDA(cudaGetLastError());
    align_traceback_kernel<int16_t><<<(n + 63) / 64, 64, 0, s>>>(utts, calls, u0, n, static_cast<int16_t *>(d_tb), src, lab,
                                                                 h->d_tid2pdf.as<int32_t>(), h->d_best.as<int32_t>(), d_ali,
                                                                 d_pdf_ids);
  } else {
    align_viterbi_kernel<int32_t><<<n, kThreads, smem, s>>>(
        utts, calls, u0, h->d_eoff.as<int32_t>(), h->d_xoff.as<int32_t>(), h->d_arcs.as<int4>(), h->d_lvl_off.as<int32_t>(),
        h->d_lvl_states.as<int32_t>(), h->d_final.as<float>(), d_ll, acoustic_scale, static_cast<int32_t *>(d_tb),
        d_tot_cost, h->d_best.as<int32_t>());
    VB_CUDA(cudaGetLastError());
    align_traceback_kernel<int32_t><<<(n + 63) / 64, 64, 0, s>>>(utts, calls, u0, n, static_cast<int32_t *>(d_tb), src, lab,
                                                                 h->d_tid2pdf.as<int32_t>(), h->d_best.as<int32_t>(), d_ali,
                                                                 d_pdf_ids);
  }
  VB_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace vb
