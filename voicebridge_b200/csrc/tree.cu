// tree.cu — tree statistics: AccumulateTreeStats (hmm/tree-accu.cc) as acc-tree-stats drives it.  For every utterance whose
// alignment SplitToPhones (hmm/hmm-utils.cc) accepts, each phone segment is taken as the central phone of an N-phone
// window; every frame of the segment adds AddStats(row, 1.0) (tree/clusterable-classes.cc) to the GaussClusterable of its
// EventType {(kPdfClass, pdf-class), (0, phone_0) ... (N-1, phone_N-1)} (only (P, central) for a context-independent central
// phone; phone 0 outside the utterance):  count += 1,  sum_x += x,  sum_x2 += x * x,  all in FP64 (x * x of a widened float
// is exact), so the results differ from the reference only by the order of the FP64 additions.
//
// Steps of one call (a packed batch of whole utterances):
//   tree_utt_kernel     a warp per utterance, over chunks of 32 frames with warp ballots and scans:
//                         IsReordered (the first transition-state change that decides it);
//                         pass 1: phone ends, in parallel form (reordered: the last non-self-loop frame at or before k is
//                         final and frame k+1 is not a self-loop, or k is last), the bad-alignment conditions OR-reduced,
//                         segment ids by a scan of the end flags, the phone of each segment from its first frame;
//                         pass 2 (good utterances): the packed 64-bit key of every frame; the first frame of a run of
//                         equal keys looks it up in (or inserts it into) the handle's hash table, the rest of the run
//                         takes that dense id by a scan.  Frames of bad utterances get id -1 and their rows are never read.
//   sort                frames counting-sorted by dense id (bin_sort_launch, shared with accum.cu / lda.cu) over the
//                       capacity-sized id range: no read-back of the key count between kernels.
//   tree_moments_kernel a CTA per (key, chunk of <= 128 of its frames): a thread per dimension sums x and x * x over the
//                       chunk in registers and flushes each with ONE FP64 atomic; thread 0 likewise for the count.
//
// The 64-bit key (private to this file): bits 0-7 pdf-class, bits 8 + 12 j .. 19 + 12 j phone at position j (0 = outside the
// utterance), bit 56 set for a context-independent central phone when N > 1 (then only position P is filled; with N = 1
// both forms are the same EventType and the same key).  Dense ids are handed out in order of first insertion; downloads
// reorder them as a std::map<EventType, ...> iterates.
#include <algorithm>
#include <numeric>
#include <utility>
#include <vector>

#include "common.h"

namespace {

// per-tid info word: phone | pdf-class << 12 | flags
constexpr uint32_t kPhoneMask = 0xFFF, kSelf = 1u << 20, kFinal = 1u << 21, kBadStart = 1u << 22, kCi = 1u << 23;
constexpr int kCiBit = 56;
constexpr int kUttWarps = 4;
constexpr int kMomThreads = 128;
constexpr unsigned long long kEmpty = ~0ull;  // no key sets bit 63
constexpr int32_t kPending = -1, kNoId = -2;   // hash slot values besides dense ids

enum { kCtrBadUtts = 0, kCtrDropped = 1, kCtrSortScratch = 2, kCtrAddDropped = 3, kCtrNumKeys = 4, kNumCtr = 5 };

__host__ __device__ inline uint64_t mix64(uint64_t z) {  // splitmix64 finaliser
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

struct Table {
  unsigned long long *keys;  // [mask + 1], kEmpty = free
  int32_t *vals;             // [mask + 1], dense id | kPending | kNoId
  unsigned long long *keys_by_id;
  unsigned long long *n_keys;
  uint32_t mask;
  int32_t max_keys;
};

// Dense id of key, inserted if new; -1 when the table has no id for it (max_keys reached, or no free slot).
__device__ int32_t find_or_insert(const Table &t, unsigned long long key) {
  uint32_t slot = (uint32_t)mix64(key) & t.mask;
  for (uint32_t probe = 0; probe <= t.mask; probe++, slot = (slot + 1) & t.mask) {
    unsigned long long k = *(volatile unsigned long long *)&t.keys[slot];
    if (k == kEmpty) {
      // a full table claims no more slots, so the probes of keys that found no room stay as short as the load factor
      // (<= 1/2) makes them; only threads racing past this check can add a slot holding kNoId
      if (*(volatile unsigned long long *)t.n_keys >= (unsigned long long)t.max_keys) return -1;
      k = atomicCAS(&t.keys[slot], kEmpty, key);
      if (k == kEmpty) {  // this thread owns the slot: hand out the next id
        const unsigned long long id = atomicAdd(t.n_keys, 1ull);
        int32_t v = kNoId;
        if (id < (unsigned long long)t.max_keys) {
          t.keys_by_id[id] = key;
          v = (int32_t)id;
        }
        __threadfence();
        atomicExch(&t.vals[slot], v);
        return v >= 0 ? v : -1;
      }
    }
    if (k == key) {  // present (perhaps being inserted by another thread right now)
      int32_t v;
      while ((v = *(volatile int32_t *)&t.vals[slot]) == kPending) __nanosleep(32);
      return v >= 0 ? v : -1;
    }
  }
  return -1;
}

__device__ __forceinline__ unsigned lanemask_le() { return 0xFFFFFFFFu >> (31 - (threadIdx.x & 31)); }

__global__ void __launch_bounds__(kUttWarps * 32) tree_utt_kernel(
    const int32_t *__restrict__ tids, const int64_t *__restrict__ fo, int32_t n_utts, const uint32_t *__restrict__ info,
    const int32_t *__restrict__ tstate, int32_t num_tids, int32_t N, int32_t P, int32_t *__restrict__ seg,
    int32_t *__restrict__ seg_phone, int32_t *__restrict__ ids, Table tab, unsigned long long *__restrict__ ctr) {
  const int lane = threadIdx.x & 31;
  const int u = blockIdx.x * kUttWarps + threadIdx.x / 32;
  if (u >= n_utts) return;
  const int64_t t0 = fo[u];
  const int n = (int)(fo[u + 1] - t0);
  const int32_t *ali = tids + t0;
  // info / transition state of frame i; an invalid transition-id makes the utterance bad (ts -1 differs from all)
  auto load = [&](int i, uint32_t &inf, int32_t &ts) -> bool {
    const int32_t tid = ali[i];
    if (tid < 1 || tid > num_tids) {
      inf = 0;
      ts = -1;
      return false;
    }
    inf = info[tid];
    ts = tstate[tid];
    return true;
  };

  // ---- IsReordered: the first i with ts(i) != ts(i+1) where one of the two is a self-loop decides
  bool reordered = false, decided = false;
  for (int base = 0; base + 1 < n && !decided; base += 32) {
    const int i = base + lane;
    bool dec = false, self_i = false;
    if (i + 1 < n) {
      uint32_t a, b;
      int32_t ta, tb;
      load(i, a, ta);
      load(i + 1, b, tb);
      self_i = a & kSelf;
      dec = ta != tb && (self_i || (b & kSelf));
    }
    const unsigned m = __ballot_sync(~0u, dec);
    if (m) {
      reordered = __shfl_sync(~0u, self_i, __ffs(m) - 1);
      decided = true;
    }
  }
  if (!decided && n > 0) {
    uint32_t a, b;
    int32_t ta, tb;
    load(0, a, ta);
    load(n - 1, b, tb);
    reordered = !(a & kSelf) && (b & kSelf);
  }

  // ---- pass 1: phone ends, badness, segment ids and phones
  bool bad = false, carry_final = false, carry_end = true;  // carry_end: "the frame before the chunk ended a phone"
  int32_t carry_seg = 0;
  for (int base = 0; base < n; base += 32) {
    const int i = base + lane;
    const bool in = i < n;
    uint32_t inf = 0, nx = 0;
    int32_t ts = 0, tn = 0;
    bool ok = true;
    if (in) {
      ok = load(i, inf, ts);
      if (i + 1 < n) ok &= load(i + 1, nx, tn);
    }
    // is the last non-self-loop frame at or before i final?
    const bool nonself = in && !(inf & kSelf);
    const unsigned ns = __ballot_sync(~0u, nonself) & lanemask_le();
    const bool fin_here = __shfl_sync(~0u, (inf & kFinal) != 0, ns ? 31 - __clz(ns) : lane);
    const bool last_final = ns ? fin_here : carry_final;
    bool end = false, b = !ok;
    if (in) {
      if (reordered ? last_final : (inf & kFinal) != 0) {
        end = !reordered || i + 1 == n || !(nx & kSelf);
      } else if (i + 1 == n) {
        end = b = true;
      } else if (ts != tn && (inf & kPhoneMask) != (nx & kPhoneMask)) {
        end = b = true;
      }
    }
    const unsigned ends = __ballot_sync(~0u, end);
    const bool prev_end = lane ? (ends >> (lane - 1)) & 1 : carry_end;
    const int32_t s = carry_seg + __popc(ends & (lanemask_le() >> 1));
    if (in) {
      seg[t0 + i] = s;
      if (prev_end) {  // first frame of segment s
        if (inf & kBadStart) b = true;
        seg_phone[t0 + s] = (int32_t)(inf & kPhoneMask) | ((inf & kCi) ? 1 << 12 : 0);
      }
    }
    bad |= __any_sync(~0u, b);
    const unsigned chunk_ns = __ballot_sync(~0u, nonself);
    if (chunk_ns) carry_final = __shfl_sync(~0u, (inf & kFinal) != 0, 31 - __clz(chunk_ns));
    carry_end = (ends >> 31) & 1;
    carry_seg += __popc(ends);
  }
  if (bad) {
    for (int i = lane; i < n; i += 32) ids[t0 + i] = -1;
    if (lane == 0) atomicAdd(&ctr[kCtrBadUtts], 1ull);
    return;
  }
  __syncwarp();  // seg / seg_phone of every lane are visible to the warp

  // ---- pass 2: packed keys, dense ids through the run heads
  const int32_t nseg = carry_seg;
  unsigned long long carry_key = kEmpty;
  int32_t carry_id = -1, dropped = 0;
  for (int base = 0; base < n; base += 32) {
    const int i = base + lane;
    const bool in = i < n;
    unsigned long long key = kEmpty;
    if (in) {
      uint32_t inf;
      int32_t ts;
      load(i, inf, ts);
      const int32_t s = seg[t0 + i], cp = seg_phone[t0 + s];
      key = (inf >> 12) & 0xFF;
      if ((cp >> 12) & 1) {  // context-independent central phone: (P, c) only
        key |= (unsigned long long)(cp & kPhoneMask) << (8 + 12 * P);
        if (N > 1) key |= 1ull << kCiBit;
      } else {
        for (int j = 0; j < N; j++) {
          const int32_t sj = s - P + j;
          const unsigned long long ph = (sj >= 0 && sj < nseg) ? (unsigned long long)(seg_phone[t0 + sj] & kPhoneMask) : 0ull;
          key |= ph << (8 + 12 * j);
        }
      }
    }
    const unsigned long long prev = __shfl_up_sync(~0u, key, 1);
    const bool head = in && key != (lane ? prev : carry_key);
    int32_t id = head ? find_or_insert(tab, key) : -1;
    const unsigned heads = __ballot_sync(~0u, head) & lanemask_le();
    const int32_t from = __shfl_sync(~0u, id, heads ? 31 - __clz(heads) : lane);
    id = heads ? from : carry_id;
    if (in) ids[t0 + i] = id;
    dropped += __popc(__ballot_sync(~0u, in && id < 0));
    carry_key = __shfl_sync(~0u, key, 31);
    carry_id = __shfl_sync(~0u, id, 31);
  }
  if (lane == 0 && dropped) atomicAdd(&ctr[kCtrDropped], (unsigned long long)dropped);
}

__global__ void __launch_bounds__(kMomThreads) tree_moments_kernel(const float *__restrict__ feats, int32_t stride,
                                                                   int32_t D, int32_t K, const int32_t *__restrict__ start,
                                                                   const int32_t *__restrict__ unit_off,
                                                                   const int32_t *__restrict__ order,
                                                                   double *__restrict__ count, double *__restrict__ sx,
                                                                   double *__restrict__ sx2) {
  __shared__ int32_t s_t[vb::kSortChunk];
  __shared__ int32_t s_k;
  const int n_units = unit_off[K + 1];
  for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
    if (threadIdx.x < 32) {  // the key of unit u: last k with unit_off[k] <= u, by a 32-way search (K is the capacity)
      int lo = 0, hi = K;
      while (hi - lo > 1) {
        const int step = (hi - lo + 31) / 32, p = lo + (int)threadIdx.x * step;
        const unsigned m = __ballot_sync(~0u, p < hi && unit_off[p] <= u);  // lane 0 (p = lo) always holds
        const int last = 31 - __clz(m);
        hi = min(hi, lo + (last + 1) * step);
        lo += last * step;
      }
      if (threadIdx.x == 0) s_k = lo;
    }
    __syncthreads();
    const int k = s_k;
    const int f0 = start[k] + (u - unit_off[k]) * vb::kSortChunk, n = min(vb::kSortChunk, start[k + 1] - f0);
    for (int i = threadIdx.x; i < n; i += blockDim.x) s_t[i] = order[f0 + i];
    __syncthreads();
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
      double a1 = 0.0, a2 = 0.0;
#pragma unroll 4
      for (int i = 0; i < n; i++) {
        const double x = (double)feats[(int64_t)s_t[i] * stride + d];
        a1 += x;
        a2 = fma(x, x, a2);
      }
      atomicAdd(&sx[(size_t)k * D + d], a1);
      atomicAdd(&sx2[(size_t)k * D + d], a2);
    }
    if (threadIdx.x == 0) atomicAdd(&count[k], (double)n);
    __syncthreads();
  }
}

// vbgpu_tree_add: a CTA per entry
__global__ void tree_add_kernel(const unsigned long long *__restrict__ keys, const double *__restrict__ cnt,
                                const double *__restrict__ ax, const double *__restrict__ ax2, int32_t D, Table tab,
                                double *__restrict__ count, double *__restrict__ sx, double *__restrict__ sx2,
                                unsigned long long *__restrict__ ctr) {
  __shared__ int32_t s_id;
  const int64_t e = blockIdx.x;
  if (threadIdx.x == 0) {
    s_id = find_or_insert(tab, keys[e]);
    if (s_id < 0) atomicAdd(&ctr[kCtrAddDropped], 1ull);
    else atomicAdd(&count[s_id], cnt[e]);
  }
  __syncthreads();
  const int32_t id = s_id;
  if (id < 0) return;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    atomicAdd(&sx[(size_t)id * D + d], ax[e * D + d]);
    atomicAdd(&sx2[(size_t)id * D + d], ax2[e * D + d]);
  }
}

Table table_of(vbgpu_tree_t h) {
  return Table{h->d_hkeys.as<unsigned long long>(), h->d_hvals.as<int32_t>(), h->d_keys_by_id.as<unsigned long long>(),
               h->d_ctr.as<unsigned long long>() + kCtrNumKeys, h->mask, h->max_keys};
}

// the EventType of a key, as sorted (key, value) pairs
std::vector<std::pair<int32_t, int32_t>> event_of(uint64_t key, int N, int P) {
  std::vector<std::pair<int32_t, int32_t>> ev;
  ev.emplace_back(-1, (int32_t)(key & 0xFF));
  const bool ci = N > 1 && ((key >> kCiBit) & 1);
  for (int j = 0; j < N; j++)
    if (!ci || j == P) ev.emplace_back(j, (int32_t)((key >> (8 + 12 * j)) & kPhoneMask));
  return ev;
}

}  // namespace

namespace vb {

int tree_check(const vbgpu_tree_opts *o, const vbgpu_tid_tables *t, int32_t dim, int32_t max_keys) {
  VB_CHECK(o && t, "null argument");
  VB_CHECK(o->context_width >= 1 && o->context_width <= 4, "context width %d outside 1 ... 4", o->context_width);
  VB_CHECK(o->central_position >= 0 && o->central_position < o->context_width, "central position %d outside [0, %d)",
           o->central_position, o->context_width);
  VB_CHECK(o->num_ci_phones >= 0 && (o->num_ci_phones == 0 || o->ci_phones), "null ci_phones");
  for (int32_t i = 1; i < o->num_ci_phones; i++) VB_CHECK(o->ci_phones[i - 1] < o->ci_phones[i], "ci_phones not sorted");
  VB_CHECK(dim >= 1 && dim <= 256, "dim %d outside 1 ... 256", dim);
  VB_CHECK(max_keys >= 1 && max_keys <= (1 << 26), "max_keys %d outside 1 ... 2^26", max_keys);
  VB_CHECK(t->num_tids >= 1, "num_tids %d < 1", t->num_tids);
  VB_CHECK(t->phone && t->hmm_state && t->pdf_class && t->trans_state && t->flags, "null transition-id table");
  for (int32_t i = 1; i <= t->num_tids; i++) {
    VB_CHECK(t->phone[i] >= 1 && t->phone[i] <= 4095, "transition-id %d: phone %d outside 1 ... 4095", i, t->phone[i]);
    VB_CHECK(t->pdf_class[i] >= 0 && t->pdf_class[i] <= 255, "transition-id %d: pdf-class %d outside 0 ... 255", i,
             t->pdf_class[i]);
    VB_CHECK(t->hmm_state[i] >= 0 && t->trans_state[i] >= 1, "transition-id %d: bad hmm-state / transition state", i);
  }
  return 0;
}

int tree_init(vbgpu_tree_t h, const vbgpu_tree_opts *o, const vbgpu_tid_tables *t) {
  h->N = o->context_width;
  h->P = o->central_position;
  h->num_tids = t->num_tids;
  std::vector<uint32_t> inf(t->num_tids + 1, 0);
  std::vector<int32_t> ts(t->num_tids + 1, 0);
  for (int32_t i = 1; i <= t->num_tids; i++) {
    const int32_t f = t->flags[i];
    uint32_t w = (uint32_t)t->phone[i] | (uint32_t)t->pdf_class[i] << 12;
    if (f & VBGPU_TID_SELF_LOOP) w |= kSelf;
    if (f & VBGPU_TID_FINAL) w |= kFinal;
    if ((f & VBGPU_TID_STATE0_EMITTING) && t->hmm_state[i] != 0) w |= kBadStart;
    if (std::binary_search(o->ci_phones, o->ci_phones + o->num_ci_phones, t->phone[i])) w |= kCi;
    inf[i] = w;
    ts[i] = t->trans_state[i];
  }
  uint32_t cap = 64;
  while (cap < 2u * (uint32_t)h->max_keys) cap <<= 1;
  h->mask = cap - 1;
  const size_t K = h->max_keys, D = h->D;
  VB_TRY(h->d_info.reserve(inf.size() * 4));
  VB_TRY(h->d_ts.reserve(ts.size() * 4));
  VB_TRY(h->d_acc.reserve(K * (1 + 2 * D) * 8));
  VB_TRY(h->d_hkeys.reserve((size_t)cap * 8));
  VB_TRY(h->d_hvals.reserve((size_t)cap * 4));
  VB_TRY(h->d_keys_by_id.reserve(K * 8));
  VB_TRY(h->d_ctr.reserve(kNumCtr * 8));
  VB_CUDA(cudaMemcpy(h->d_info.p, inf.data(), inf.size() * 4, cudaMemcpyHostToDevice));
  VB_CUDA(cudaMemcpy(h->d_ts.p, ts.data(), ts.size() * 4, cudaMemcpyHostToDevice));
  return tree_zero(h, h->stream);
}

int tree_zero(vbgpu_tree_t h, cudaStream_t s) {
  const size_t K = h->max_keys, D = h->D, cap = (size_t)h->mask + 1;
  VB_CUDA(cudaMemsetAsync(h->d_acc.p, 0, K * (1 + 2 * D) * 8, s));
  VB_CUDA(cudaMemsetAsync(h->d_hkeys.p, 0xFF, cap * 8, s));  // kEmpty
  VB_CUDA(cudaMemsetAsync(h->d_hvals.p, 0xFF, cap * 4, s));  // kPending
  VB_CUDA(cudaMemsetAsync(h->d_ctr.p, 0, kNumCtr * 8, s));
  VB_CUDA(cudaStreamSynchronize(s));
  return 0;
}

int tree_launch(vbgpu_tree_t h, const float *d_feats, int32_t stride, const int32_t *d_tids, const int64_t *d_fo,
                int32_t n_utts, int64_t T, cudaStream_t s) {
  if (n_utts == 0) return 0;
  VB_CHECK(T < ((int64_t)1 << 31), "more than 2^31 frames in one call");
  const size_t tb = (size_t)std::max<int64_t>(T, 1) * 4;
  VB_TRY(h->d_seg.reserve(tb));
  VB_TRY(h->d_seg_phone.reserve(tb));
  VB_TRY(h->d_ids.reserve(tb));
  unsigned long long *ctr = h->d_ctr.as<unsigned long long>();
  tree_utt_kernel<<<(n_utts + kUttWarps - 1) / kUttWarps, kUttWarps * 32, 0, s>>>(
      d_tids, d_fo, n_utts, h->d_info.as<uint32_t>(), h->d_ts.as<int32_t>(), h->num_tids, h->N, h->P, h->d_seg.as<int32_t>(),
      h->d_seg_phone.as<int32_t>(), h->d_ids.as<int32_t>(), table_of(h), ctr);
  VB_CUDA(cudaGetLastError());
  if (T == 0) return 0;

  const int K = h->max_keys, D = h->D;
  double *count = h->d_acc.as<double>(), *sx = count + K, *sx2 = sx + (size_t)K * D;
  BinSort bs;
  VB_TRY(bin_sort_launch(h->d_ids.as<int32_t>(), T, K, nullptr, h->device, &h->d_work, ctr + kCtrSortScratch, s, &bs));
  const int64_t max_units = (int64_t)K + T / kSortChunk + 1;
  const int grid = (int)std::min<int64_t>(max_units, (int64_t)num_sms(h->device) * 16);
  const int threads = std::min(kMomThreads, (D + 31) / 32 * 32);
  tree_moments_kernel<<<grid, threads, 0, s>>>(d_feats, stride, D, K, bs.start, bs.unit_off, bs.order, count, sx, sx2);
  VB_CUDA(cudaGetLastError());
  return 0;
}

int tree_counters(vbgpu_tree_t h, int64_t *bad_utts, int64_t *dropped, int64_t *num_keys, bool reset) {
  unsigned long long c[kNumCtr];
  VB_CUDA(cudaMemcpy(c, h->d_ctr.p, sizeof(c), cudaMemcpyDeviceToHost));
  if (bad_utts) *bad_utts = (int64_t)c[kCtrBadUtts];
  if (dropped) *dropped = (int64_t)c[kCtrDropped];
  if (num_keys) *num_keys = (int64_t)std::min<unsigned long long>(c[kCtrNumKeys], (unsigned long long)h->max_keys);
  if (reset) VB_CUDA(cudaMemset(h->d_ctr.p, 0, 2 * 8));  // the bad-utterance and dropped-frame counts only
  return 0;
}

int tree_download(vbgpu_tree_t h, int32_t *pdf_class, int32_t *phones, double *count, double *sum_x, double *sum_x2) {
  int64_t K64 = 0;
  VB_TRY(tree_counters(h, nullptr, nullptr, &K64, false));
  const size_t K = (size_t)K64, D = h->D, N = h->N, cap = h->max_keys;
  std::vector<unsigned long long> keys(K);
  std::vector<double> c(K), a(K * D), b(K * D);
  const double *acc = h->d_acc.as<double>();
  if (K) {
    VB_CUDA(cudaMemcpy(keys.data(), h->d_keys_by_id.p, K * 8, cudaMemcpyDeviceToHost));
    VB_CUDA(cudaMemcpy(c.data(), acc, K * 8, cudaMemcpyDeviceToHost));
    VB_CUDA(cudaMemcpy(a.data(), acc + cap, K * D * 8, cudaMemcpyDeviceToHost));
    VB_CUDA(cudaMemcpy(b.data(), acc + cap + cap * D, K * D * 8, cudaMemcpyDeviceToHost));
  }
  std::vector<std::vector<std::pair<int32_t, int32_t>>> ev(K);
  for (size_t k = 0; k < K; k++) ev[k] = event_of(keys[k], h->N, h->P);
  std::vector<size_t> ord(K);
  std::iota(ord.begin(), ord.end(), 0);
  std::sort(ord.begin(), ord.end(), [&](size_t x, size_t y) { return ev[x] < ev[y]; });  // std::map<EventType, ...> order
  for (size_t r = 0; r < K; r++) {
    const size_t k = ord[r];
    if (pdf_class) pdf_class[r] = ev[k][0].second;
    if (phones) {
      for (size_t j = 0; j < N; j++) phones[r * N + j] = -1;
      for (size_t q = 1; q < ev[k].size(); q++) phones[r * N + ev[k][q].first] = ev[k][q].second;
    }
    if (count) count[r] = c[k];
    if (sum_x) std::copy(a.begin() + k * D, a.begin() + (k + 1) * D, sum_x + r * D);
    if (sum_x2) std::copy(b.begin() + k * D, b.begin() + (k + 1) * D, sum_x2 + r * D);
  }
  return 0;
}

int tree_add(vbgpu_tree_t h, int32_t n, const int32_t *pdf_class, const int32_t *phones, const double *count,
             const double *sum_x, const double *sum_x2, int64_t *dropped) {
  const int N = h->N, P = h->P;
  const size_t D = h->D;
  std::vector<unsigned long long> keys(n);
  for (int32_t e = 0; e < n; e++) {
    const int32_t *ph = phones + (size_t)e * N;
    VB_CHECK(pdf_class[e] >= 0 && pdf_class[e] <= 255, "entry %d: pdf-class %d outside 0 ... 255", e, pdf_class[e]);
    int present = 0;
    for (int j = 0; j < N; j++) {
      VB_CHECK(ph[j] >= -1 && ph[j] <= 4095, "entry %d: phone %d outside -1 ... 4095", e, ph[j]);
      present += ph[j] >= 0;
    }
    unsigned long long key = (unsigned long long)pdf_class[e];
    if (present == N) {
      for (int j = 0; j < N; j++) key |= (unsigned long long)ph[j] << (8 + 12 * j);
    } else {
      VB_CHECK(present == 1 && ph[P] >= 0, "entry %d: neither a full context nor the central position alone", e);
      key |= (unsigned long long)ph[P] << (8 + 12 * P) | 1ull << kCiBit;
    }
    keys[e] = key;
  }
  if (n == 0) return 0;
  cudaStream_t s = h->stream;
  const size_t kb = (size_t)n * 8, vb_ = (size_t)n * D * 8;
  VB_TRY(h->d_stage.reserve(kb * 2 + 2 * vb_));
  char *st = h->d_stage.as<char>();
  unsigned long long *d_keys = reinterpret_cast<unsigned long long *>(st);
  double *d_cnt = reinterpret_cast<double *>(st + kb), *d_x = d_cnt + n, *d_x2 = d_x + (size_t)n * D;
  VB_CUDA(cudaMemcpyAsync(d_keys, keys.data(), kb, cudaMemcpyHostToDevice, s));
  VB_CUDA(cudaMemcpyAsync(d_cnt, count, kb, cudaMemcpyHostToDevice, s));
  VB_CUDA(cudaMemcpyAsync(d_x, sum_x, vb_, cudaMemcpyHostToDevice, s));
  VB_CUDA(cudaMemcpyAsync(d_x2, sum_x2, vb_, cudaMemcpyHostToDevice, s));
  unsigned long long *ctr = h->d_ctr.as<unsigned long long>();
  VB_CUDA(cudaMemsetAsync(ctr + kCtrAddDropped, 0, 8, s));
  const size_t K = h->max_keys;
  double *c = h->d_acc.as<double>();
  tree_add_kernel<<<n, std::min(kMomThreads, (int)(D + 31) / 32 * 32), 0, s>>>(d_keys, d_cnt, d_x, d_x2, (int32_t)D,
                                                                              table_of(h), c, c + K, c + K + K * D, ctr);
  VB_CUDA(cudaGetLastError());
  unsigned long long dr = 0;
  VB_CUDA(cudaMemcpyAsync(&dr, ctr + kCtrAddDropped, 8, cudaMemcpyDeviceToHost, s));
  VB_CUDA(cudaStreamSynchronize(s));
  *dropped = (int64_t)dr;
  return 0;
}

}  // namespace vb
