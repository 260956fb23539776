// decode.cu — one-best decoding: the beam search of gmm-decode-faster (FasterDecoder::Decode / ReachedFinal /
// GetBestPath) over one decoding graph (HCLG) that every utterance of a packed batch shares.  Semantics, prune rule,
// tie rules and limits are stated in include/vbgpu.h (vbgpu_decoder_*).
//
// Create time (host): the graph is checked, then laid out for the kernels —
//   * the outgoing arcs of every state, emitting ones and epsilon ones in two CSR lists by source, each arc stored as
//     {dst, column (per call), weight, original arc index} in original arc order;
//   * the epsilon levels: level(s) = the longest epsilon path into s (Kahn's topological sort, which also finds cycles).
//     Pushing the epsilon arcs out of the tokens of level 0, then 1, ... relaxes the closure exactly, as align.cu's pull
//     over the same levels does.
// Call time: decode_cols_kernel writes the model's column of every emitting arc, then per group of utterances
//   decode_search_kernel     a CTA per utterance loops over the frames.  The token set lives in global memory: a dense
//                            state -> slot map and a dense FP64 cost key over S (reset only where touched), and per slot
//                            its state, cost and back-pointer.  A relaxation is three passes over the arcs: a 64-bit
//                            atomicMin on the order-preserving key of the cost (and the slot allocation), an atomicMin on
//                            the back-pointer code among the arcs with exactly that cost (lowest arc index), and a commit
//                            per slot.  Arcs are spread over threads by a CTA-wide prefix sum of out-degrees.  The
//                            max_active cutoff is a radix select over the slots' cost keys.  Before each frame the
//                            survivors of the prune are recorded: previous-frame record, emitting arc, epsilon chain.
//   decode_traceback_kernel  a thread per utterance walks the best token's chain and the records back to the start
//                            state and writes transition-ids, pdf-ids and words.
// Lattice form (vbgpu_decode_lattice*): decode_search_kernel<true> also keeps every frame's tokens and links in the
// utterance's lattice store (Lat), pruned at each frame to what can still reach the next frame, and
//   decode_lattice_kernel    a CTA per utterance runs the exact final prune backwards over the store and writes the
//                            numbered lattice.
#include <algorithm>
#include <cmath>
#include <vector>

#include "common.h"

namespace {

// 256 threads per utterance; __launch_bounds__(kThreads, 4) leaves room for four CTAs per SM.
constexpr int kThreads = 256, kWarps = kThreads / 32;
constexpr unsigned long long kNone = ~0ull;                   // no back-pointer (the start token) / no candidate
constexpr unsigned long long kKeyInf = 0xFFF0000000000000ull;  // key(+inf)
constexpr unsigned long long kEps = 1ull << 63;                // back-pointer code of an epsilon arc

// Order-preserving key of an FP64 cost (NaN never reaches it) and back.
__device__ __forceinline__ unsigned long long key_of(double c) {
  const long long b = __double_as_longlong(c);
  return b < 0 ? ~(unsigned long long)b : (unsigned long long)b | (1ull << 63);
}
__device__ __forceinline__ double cost_of(unsigned long long k) {
  return __longlong_as_double((long long)((k >> 63) ? (k & ~(1ull << 63)) : ~k));
}

struct Smem {
  int off[kThreads], a0[kThreads], warp[kWarps];
  unsigned int hist[256];
  unsigned long long red;
  unsigned long long prefix;
  int kk, n, m, over;
  int lover, lblock, ltop, ttop, lpeak;  // lattice: store full, links of the current frame, link / token tops, peak
};

__device__ unsigned long long block_min(unsigned long long v, Smem &sh) {
  for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();  // earlier readers of sh.red are done
  if (threadIdx.x == 0) sh.red = kNone;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) atomicMin(&sh.red, v);
  __syncthreads();
  return sh.red;
}

// Exclusive prefix sum of one int per thread; *total gets the sum.
__device__ int block_scan(int v, Smem &sh, int *total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int x = v;
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) sh.warp[w] = x;
  __syncthreads();
  int base = 0, tot = 0;
  for (int i = 0; i < kWarps; i++) {
    base += i < w ? sh.warp[i] : 0;
    tot += sh.warp[i];
  }
  *total = tot;
  return base + x - v;
}

// The k-th smallest (1-based, k <= n) of keys[0, n): most significant byte first, a 256-bin histogram per byte.
__device__ unsigned long long radix_select(const unsigned long long *keys, int n, int k, Smem &sh) {
  if (threadIdx.x == 0) sh.prefix = 0, sh.kk = k;
  for (int shift = 56; shift >= 0; shift -= 8) {
    for (int b = threadIdx.x; b < 256; b += kThreads) sh.hist[b] = 0;
    __syncthreads();
    const unsigned long long mask = shift == 56 ? 0ull : ~0ull << (shift + 8), prefix = sh.prefix;
    for (int i = threadIdx.x; i < n; i += kThreads) {
      const unsigned long long v = keys[i];
      if ((v & mask) == prefix) atomicAdd(&sh.hist[(v >> shift) & 255], 1u);
    }
    __syncthreads();
    if (threadIdx.x < 32) {  // one warp: lane l owns bins 8l ... 8l + 7
      const int lane = threadIdx.x;
      unsigned int own = 0;
      for (int b = 0; b < 8; b++) own += sh.hist[lane * 8 + b];
      unsigned int inc = own;
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned int y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
      }
      const int kk = sh.kk;
      const unsigned int hit = __ballot_sync(0xffffffffu, inc >= (unsigned)kk);
      if (lane == __ffs(hit) - 1) {
        unsigned int before = inc - own;
        int b = lane * 8;
        while (before + sh.hist[b] < (unsigned)kk) before += sh.hist[b++];
        sh.prefix = prefix | ((unsigned long long)b << shift);
        sh.kk = kk - (int)before;
      }
    }
    __syncthreads();
  }
  return sh.prefix;
}

// Calls work(source, arc, pos) for every outgoing arc of sources [0, n_src): range(i, &a0, &deg) gives source i's
// arcs, pos numbers the arcs of all sources in source order from 0.  Returns the number of arcs.
template <class Range, class Work>
__device__ int for_each_arc(int n_src, Range range, Work work, Smem &sh) {
  int pos0 = 0;
  for (int base = 0; base < n_src; base += kThreads) {
    int a0 = 0, deg = 0;
    if (base + threadIdx.x < n_src) range(base + threadIdx.x, &a0, &deg);
    int total;
    const int ex = block_scan(deg, sh, &total);
    sh.off[threadIdx.x] = ex;
    sh.a0[threadIdx.x] = a0;
    __syncthreads();
    const int cnt = min(kThreads, n_src - base);
    for (int j = threadIdx.x; j < total; j += kThreads) {
      int lo = 0, hi = cnt;  // the last source whose offset is <= j
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (sh.off[mid] <= j) lo = mid;
        else hi = mid;
      }
      work(base + lo, sh.a0[lo] + j - sh.off[lo], pos0 + j);
    }
    pos0 += total;
    __syncthreads();
  }
  return pos0;
}

struct Utt {  // the workspace of one utterance (vb::decode_ws_bytes)
  unsigned long long *key;  // [S] cost key of the state in the current set, kKeyInf when absent
  int32_t *map;             // [S] slot of the state in the current set, -1 when absent
  unsigned long long *kb, *win, *wn;  // [cap] per slot: cost key at the last commit, back-pointer, candidate
  int32_t *st, *src;                  // [cap] per slot: state; the sources of an epsilon pass
  double *s_cost;                     // [cap2] survivors: cost
  int32_t *s_st;                      //        state
  int32_t *rec;                       // [T][cap2][2 + L] survivor records
};

__device__ __forceinline__ void carve(Utt &w, unsigned char *p, int S, int cap, int cap2) {
  auto take = [&](size_t bytes) {
    unsigned char *q = p;
    p += (bytes + 15) & ~size_t(15);
    return q;
  };
  w.key = reinterpret_cast<unsigned long long *>(take((size_t)S * 8));
  w.kb = reinterpret_cast<unsigned long long *>(take((size_t)cap * 8));
  w.win = reinterpret_cast<unsigned long long *>(take((size_t)cap * 8));
  w.wn = reinterpret_cast<unsigned long long *>(take((size_t)cap * 8));
  w.s_cost = reinterpret_cast<double *>(take((size_t)cap2 * 8));
  w.map = reinterpret_cast<int32_t *>(take((size_t)S * 4));
  w.st = reinterpret_cast<int32_t *>(take((size_t)cap * 4));
  w.src = reinterpret_cast<int32_t *>(take((size_t)cap * 4));
  w.s_st = reinterpret_cast<int32_t *>(take((size_t)cap2 * 4));
  w.rec = reinterpret_cast<int32_t *>(p);
}

// The lattice store of one utterance (vb::lattice_arena_bytes): the tokens and links of every frame, as each prune
// keeps them.  A link is {source token, destination token, original arc index | kEpsLink, acoustic cost bits}.  Until
// the prune of frame f, the links into frame f hold slots of the current set where they name frame f's tokens.
constexpr int kEpsLink = (int)0x80000000;
struct Lat {
  double *alpha;                          // [NT] per token: cost
  unsigned long long *extra, *key;        // [NT] lattice pass: extra cost key; (level, state) key
  int32_t *state, *num, *e_first, *x_first, *abase, *ord;  // [NT] graph state; lattice pass: number, link runs ...
  int4 *link;                             // [NL]
  int32_t *keep;                          // [NL] lattice pass: kept by the final prune
  int32_t *tid;                           // [cap] per slot: kept flag, then token index (-1: dropped)
  int32_t *s_tok;                         // [cap2] per survivor: slot, then token index
  int32_t *f_tok, *f_lnk;                 // [T + 2] frame f's tokens [f_tok[f], f_tok[f+1]), links into it likewise
  int NT, NL;
};

__device__ __forceinline__ void carve_lat(Lat &L, unsigned char *p, int NT, int NL, int cap, int cap2, int64_t T) {
  auto take = [&](size_t bytes) {
    unsigned char *q = p;
    p += (bytes + 15) & ~size_t(15);
    return q;
  };
  L.NT = NT, L.NL = NL;
  L.alpha = reinterpret_cast<double *>(take((size_t)NT * 8));
  L.extra = reinterpret_cast<unsigned long long *>(take((size_t)NT * 8));
  L.key = reinterpret_cast<unsigned long long *>(take((size_t)NT * 8));
  L.link = reinterpret_cast<int4 *>(take((size_t)NL * 16));
  int32_t **ints[] = {&L.state, &L.num, &L.e_first, &L.x_first, &L.abase, &L.ord};
  for (int32_t **q : ints) *q = reinterpret_cast<int32_t *>(take((size_t)NT * 4));
  L.keep = reinterpret_cast<int32_t *>(take((size_t)NL * 4));
  L.tid = reinterpret_cast<int32_t *>(take((size_t)cap * 4));
  L.s_tok = reinterpret_cast<int32_t *>(take((size_t)cap2 * 4));
  L.f_tok = reinterpret_cast<int32_t *>(take((size_t)(T + 2) * 4));
  L.f_lnk = reinterpret_cast<int32_t *>(take((size_t)(T + 2) * 4));
}

// One relaxation of the arcs out of n_src sources into the current set (emitting step or one epsilon level):
// cost(i, a) is the candidate cost through arc position a of source i (NaN / +inf: no candidate), code(i, a) its
// back-pointer code.  Returns false when the set outgrew its capacity.  kLat: every arc is also recorded as a link,
// link(i, a) giving its {source, acoustic cost bits}; a store without room for them ends the lattice (sh.lover).
template <bool kLat, class Range, class Cost, class Code, class Link>
__device__ bool relax(int n_src, Range range, Cost cost, Code code, Link link, int eps_bit,
                      const int4 *__restrict__ arcs, Utt &w, Lat &L, int cap, Smem &sh) {
  const int total = for_each_arc(n_src, range, [&](int i, int a, int) {
    const double v = cost(i, a);
    if (!(v < INFINITY)) return;
    const int d = __ldg(arcs + a).x;
    atomicMin(w.key + d, key_of(v));
    if (*(volatile int32_t *)(w.map + d) == -1 && atomicCAS(w.map + d, -1, -2) == -1) {
      const int k = atomicAdd(&sh.n, 1);
      if (k < cap) {
        w.st[k] = d, w.kb[k] = kKeyInf, w.win[k] = kNone, w.wn[k] = kNone;
        w.map[d] = k;
      } else {
        sh.over = 1;
      }
    }
  }, sh);
  if (sh.over) return false;
  const int lb = kLat ? sh.ltop : 0;
  const bool rec = kLat && !sh.lover && (long long)lb + total <= L.NL;
  for_each_arc(n_src, range, [&](int i, int a, int pos) {  // of the arcs that reach the minimum, the lowest code
    const double v = cost(i, a);
    const int4 A = __ldg(arcs + a);
    if (rec) {
      const int2 sl = link(i, a);
      L.link[lb + pos] = make_int4(sl.x, v < INFINITY ? w.map[A.x] : -1, A.w | eps_bit, sl.y);
    }
    if (!(v < INFINITY)) return;
    if (key_of(v) == w.key[A.x]) atomicMin(w.wn + w.map[A.x], code(i, a));
  }, sh);
  if (kLat && threadIdx.x == 0) {
    if (rec) sh.ltop = lb + total, sh.lpeak = max(sh.lpeak, lb + total);
    else sh.lover = 1;
  }
  const int n = sh.n;
  for (int k = threadIdx.x; k < n; k += kThreads) {  // commit: a lower cost takes the new back-pointer, an equal one
    const unsigned long long c = w.wn[k];           // keeps the lower code (emitting codes sort before epsilon ones)
    if (c == kNone) continue;
    const unsigned long long key = w.key[w.st[k]];
    w.win[k] = key < w.kb[k] ? c : min(w.win[k], c);
    w.kb[k] = key;
    w.wn[k] = kNone;
  }
  __syncthreads();
  return true;
}

// Epsilon closure of the current set, level after level, out of tokens whose cost is below cut.
template <bool kLat>
__device__ bool closure(const vb::DecodeArgs &g, Utt &w, Lat &L, double cut, Smem &sh) {
  for (int l = 0; l < g.n_lvls; l++) {
    if (threadIdx.x == 0) sh.m = 0;
    __syncthreads();
    const int n = sh.n;
    for (int k = threadIdx.x; k < n; k += kThreads) {
      const int s = w.st[k];
      if (__ldg(g.lvl + s) == l && __ldg(g.x_off + s + 1) > __ldg(g.x_off + s) && cost_of(w.kb[k]) < cut)
        w.src[atomicAdd(&sh.m, 1)] = k;
    }
    __syncthreads();
    const int m = sh.m;
    if (m == 0) continue;
    const bool ok = relax<kLat>(
        m,
        [&](int i, int *a0, int *deg) {
          const int s = w.st[w.src[i]];
          *a0 = __ldg(g.x_off + s);
          *deg = __ldg(g.x_off + s + 1) - *a0;
        },
        [&](int i, int a) { return cost_of(w.kb[w.src[i]]) + (double)__int_as_float(__ldg(g.x_arcs + a).z); },
        [&](int i, int a) {
          return kEps | ((unsigned long long)__ldg(g.x_arcs + a).w << 32) | (unsigned)w.src[i];
        },
        [&](int i, int) { return make_int2(w.src[i], 0); }, kEpsLink, g.x_arcs, w, L, g.cap, sh);
    if (!ok) return false;
  }
  return true;
}

// Lattice, at the prune of frame t (n tokens in the current set, L.tid[k] = 1 for the tokens it expands, ns survivors
// with L.s_tok[j] = their slot) or after the last frame (every token marked, ns = 0): also marks the tokens with an
// epsilon path to a marked one (levels from the highest down: epsilon arcs go to higher levels), stores the marked
// tokens as frame t's, and compacts the links into frame t in order, dropping those into unmarked tokens.
__device__ void lat_keep(const vb::DecodeArgs &g, Utt &w, Lat &L, int n, int ns, int64_t t, Smem &sh) {
  if (sh.lover) return;
  const int lb = sh.lblock, le = sh.ltop;
  for (int l = g.n_lvls - 1; l >= 0; l--) {
    for (int i = lb + threadIdx.x; i < le; i += kThreads) {
      const int4 k = L.link[i];
      if (k.z < 0 && k.y >= 0 && L.tid[k.y] && __ldg(g.lvl + w.st[k.x]) == l) L.tid[k.x] = 1;
    }
    __syncthreads();
  }
  int top = sh.ttop;
  for (int c = 0; c < n; c += kThreads) {
    const int k = c + threadIdx.x, keep = k < n && L.tid[k];
    int total;
    const int j = top + block_scan(keep, sh, &total);
    if (keep && j < L.NT) L.alpha[j] = cost_of(w.kb[k]), L.state[j] = w.st[k];
    if (k < n) L.tid[k] = keep ? j : -1;
    top += total;
    __syncthreads();
  }
  if (top > L.NT) {
    if (threadIdx.x == 0) sh.lover = 1;
    __syncthreads();
    return;
  }
  int lo = lb;
  for (int c = lb; c < le; c += kThreads) {
    const int i = c + threadIdx.x;
    int4 k = i < le ? L.link[i] : make_int4(0, -1, 0, 0);
    int d = k.y >= 0 ? L.tid[k.y] : -1;
    if (d >= 0) {  // (the marking keeps the source of a link into a kept token; a dropped one drops the link)
      k.y = d;
      if (k.z < 0) k.x = L.tid[k.x], d = k.x >= 0 ? d : -1;
    }
    int total;
    const int j = lo + block_scan(d >= 0, sh, &total);  // every thread has read its link
    if (d >= 0) L.link[j] = k;
    lo += total;
    __syncthreads();
  }
  for (int j = threadIdx.x; j < ns; j += kThreads) L.s_tok[j] = L.tid[L.s_tok[j]];
  if (threadIdx.x == 0) {
    L.f_tok[t + 1] = top, L.f_lnk[t + 1] = lo;
    sh.ttop = top, sh.ltop = lo, sh.lblock = lo;
  }
  __syncthreads();
}

// kLat: the lattice form, which also records tokens and links in the utterance's lattice store (Lat).
template <bool kLat>
__global__ void __launch_bounds__(kThreads, 4) decode_search_kernel(vb::DecodeArgs g, int32_t u0) {
  __shared__ Smem sh;
  const int u = u0 + blockIdx.x;
  const vb::DecodeCall C = g.calls[u];
  const int S = g.S, cap = g.cap, cap2 = g.cap2, RW = 2 + g.n_lvls;
  Utt w;
  carve(w, g.ws + C.ws_off, S, cap, cap2);
  Lat L{};
  if (kLat) carve_lat(L, g.ws + C.lat_off, C.NT, C.NL, cap, cap2, C.T);
  for (int s = threadIdx.x; s < S; s += kThreads) w.key[s] = kKeyInf, w.map[s] = -1;
  __syncthreads();
  if (threadIdx.x == 0) {
    sh.n = 1, sh.over = 0;
    sh.lover = 0, sh.lblock = 0, sh.ltop = 0, sh.ttop = 0, sh.lpeak = 0;
    if (kLat) L.f_tok[0] = 0, L.f_lnk[0] = 0;
    w.st[0] = g.start, w.kb[0] = key_of(0.0), w.win[0] = kNone, w.wn[0] = kNone;
    w.key[g.start] = key_of(0.0), w.map[g.start] = 0;
  }
  __syncthreads();
  int status = closure<kLat>(g, w, L, INFINITY, sh) ? 0 : 3;
  for (int64_t t = 0; t < C.T && status == 0; t++) {
    // prune: cutoff c1 + beam, lowered to c_(max_active + 1) when the set is larger; the best token always survives
    const int n = sh.n;
    unsigned long long kmin = kNone;
    for (int k = threadIdx.x; k < n; k += kThreads) kmin = min(kmin, w.kb[k]);
    kmin = block_min(kmin, sh);
    const double c1 = cost_of(kmin);
    double cut = c1 + (double)g.beam;
    if (n > g.max_active) {
      const double ck = cost_of(radix_select(w.kb, n, g.max_active + 1, sh));
      cut = ck < cut ? ck : cut;
    }
    if (threadIdx.x == 0) sh.m = 0;
    if (kLat)
      for (int k = threadIdx.x; k < n; k += kThreads) L.tid[k] = 0;
    __syncthreads();
    int32_t *row = w.rec + t * cap2 * RW;
    for (int k = threadIdx.x; k < n; k += kThreads) {
      const double c = cost_of(w.kb[k]);
      if (!(c < cut || w.kb[k] == kmin)) continue;
      const int j = atomicAdd(&sh.m, 1);
      if (j >= cap2) continue;
      if (kLat) L.tid[k] = 1, L.s_tok[j] = k;
      w.s_st[j] = w.st[k], w.s_cost[j] = c;
      int32_t *r = row + (int64_t)j * RW;  // the survivor's epsilon chain, newest arc first, then its emitting arc
      int x = k, e = 0;
      unsigned long long b = w.win[x];
      while (b != kNone && (b & kEps)) {
        r[2 + e++] = (int)((b >> 32) & 0x7fffffff);
        x = (int)(unsigned)b;
        b = w.win[x];
      }
      for (; e < g.n_lvls; e++) r[2 + e] = -1;
      r[0] = b == kNone ? -1 : (int)(unsigned)b;
      r[1] = b == kNone ? -1 : (int)(b >> 32);
    }
    __syncthreads();
    const int ns = sh.m;
    if (ns > cap2) {
      status = 3;
      break;
    }
    if (kLat) lat_keep(g, w, L, n, ns, t, sh);
    for (int k = threadIdx.x; k < n; k += kThreads) w.key[w.st[k]] = kKeyInf, w.map[w.st[k]] = -1;
    __syncthreads();
    if (threadIdx.x == 0) sh.n = 0;
    __syncthreads();
    // emitting step of frame t
    const float *llr = g.ll + (C.ll_row0 + t) * g.ll_stride;
    const bool ok = relax<kLat>(
        ns,
        [&](int i, int *a0, int *deg) {
          const int s = w.s_st[i];
          *a0 = __ldg(g.e_off + s);
          *deg = __ldg(g.e_off + s + 1) - *a0;
        },
        [&](int i, int a) {
          const int4 A = __ldg(g.e_arcs + a);
          const float ac = -__fmul_rn(g.scale, __ldg(llr + A.y));
          return (w.s_cost[i] + (double)__int_as_float(A.z)) + (double)ac;
        },
        [&](int i, int a) { return ((unsigned long long)__ldg(g.e_arcs + a).w << 32) | (unsigned)i; },
        [&](int i, int a) {
          return make_int2(L.s_tok[i], __float_as_int(-__fmul_rn(g.scale, __ldg(llr + __ldg(g.e_arcs + a).y))));
        },
        0, g.e_arcs, w, L, cap, sh);
    if (!ok) {
      status = 3;
      break;
    }
    const int n1 = sh.n;
    if (n1 == 0) {
      status = 2;
      break;
    }
    unsigned long long bmin = kNone;
    for (int k = threadIdx.x; k < n1; k += kThreads) bmin = min(bmin, w.kb[k]);
    bmin = block_min(bmin, sh);
    if (!closure<kLat>(g, w, L, cost_of(bmin) + (double)g.beam, sh)) status = 3;
  }
  if (kLat) {
    if (status == 0) {  // the last frame's tokens are all kept until the final prune
      for (int k = threadIdx.x; k < sh.n; k += kThreads) L.tid[k] = 1;
      __syncthreads();
      lat_keep(g, w, L, sh.n, 0, C.T, sh);
    }
    if (threadIdx.x == 0) {
      g.lat.lattice_status[u] = sh.lover;
      if (g.lat.arena_peak) g.lat.arena_peak[2 * u] = sh.ttop, g.lat.arena_peak[2 * u + 1] = sh.lpeak;
    }
  }
  // end: the best cost + final (status 0), else the best cost (status 1); equal values go to the lower state
  const int n = sh.n;
  unsigned long long best = kNone;
  if (status == 0) {
    for (int k = threadIdx.x; k < n; k += kThreads) {
      const float f = __ldg(g.finals + w.st[k]);
      if (f < INFINITY) best = min(best, key_of(cost_of(w.kb[k]) + (double)f));
    }
    best = block_min(best, sh);
    if (best == kNone) {
      status = 1;
      for (int k = threadIdx.x; k < n; k += kThreads) best = min(best, w.kb[k]);
      best = block_min(best, sh);
    }
    unsigned long long bs = kNone;
    for (int k = threadIdx.x; k < n; k += kThreads) {
      const float f = __ldg(g.finals + w.st[k]);
      const unsigned long long v = status == 0 ? (f < INFINITY ? key_of(cost_of(w.kb[k]) + (double)f) : kNone) : w.kb[k];
      if (v == best) bs = min(bs, (unsigned long long)w.st[k]);
    }
    bs = block_min(bs, sh);
    if (threadIdx.x == 0) g.best[u] = w.map[(int)bs];
  }
  if (threadIdx.x == 0) {
    g.status[u] = status;
    g.tot_cost[u] = status <= 1 ? cost_of(best) : INFINITY;
  }
}

// A thread per utterance: the best token's epsilon chain in the final set, then the survivor records from row T - 1
// back to row 0.  Pass 0 counts the words, pass 1 writes them from the last one back.
__global__ void __launch_bounds__(64) decode_traceback_kernel(vb::DecodeArgs g, int32_t u0, int32_t n_utts,
                                                              const int32_t *__restrict__ a_ilabel,
                                                              const int32_t *__restrict__ a_olabel,
                                                              const int32_t *__restrict__ tid2pdf) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_utts) return;
  const int u = u0 + i;
  const vb::DecodeCall C = g.calls[u];
  int32_t *ali = g.ali + C.f0, *pdf = g.pdf_ids ? g.pdf_ids + C.f0 : nullptr;
  if (g.status[u] >= 2) {
    for (int64_t t = 0; t < C.T; t++) {
      ali[t] = 0;
      if (pdf) pdf[t] = -1;
    }
    g.num_words[u] = 0;
    return;
  }
  Utt w;
  carve(w, g.ws + C.ws_off, g.S, g.cap, g.cap2);
  const int RW = 2 + g.n_lvls;
  int32_t *words = g.words + (int64_t)u * g.max_words;
  int nw = 0;
  for (int pass = 0; pass < 2; pass++) {
    int k = nw;
    auto word = [&](int a) {
      const int ol = __ldg(a_olabel + a);
      if (!ol) return;
      if (pass == 0) nw++;
      else if (--k < g.max_words) words[k] = ol;
    };
    auto emit = [&](int a, int64_t t) {
      if (pass) {
        const int lab = __ldg(a_ilabel + a);
        ali[t] = lab;
        if (pdf) pdf[t] = __ldg(tid2pdf + lab);
      }
      word(a);
    };
    int x = g.best[u];
    unsigned long long b = w.win[x];
    while (b != kNone && (b & kEps)) {
      word((int)((b >> 32) & 0x7fffffff));
      x = (int)(unsigned)b;
      b = w.win[x];
    }
    if (b == kNone) continue;  // T = 0
    int64_t r = C.T - 1;
    emit((int)(b >> 32), r);
    int j = (int)(unsigned)b;
    for (;;) {
      const int32_t *R = w.rec + (r * g.cap2 + j) * RW;
      for (int e = 0; e < g.n_lvls && R[2 + e] >= 0; e++) word(R[2 + e]);
      if (R[1] < 0) break;
      emit(R[1], r - 1);
      j = R[0];
      r--;
    }
  }
  g.num_words[u] = nw;
}

// A CTA per utterance, after the search: the exact final prune of the lattice store, then the numbered output.
__global__ void __launch_bounds__(kThreads) decode_lattice_kernel(vb::DecodeArgs g, int32_t u0) {
  __shared__ Smem sh;
  __shared__ unsigned long long tile[kThreads];
  const int u = u0 + blockIdx.x;
  const vb::DecodeCall C = g.calls[u];
  const vbgpu_lattice_out &o = g.lat;
  const int status = g.status[u];
  if (status >= 2 || o.lattice_status[u] != 0) {  // an empty lattice / a store that overflowed
    if (threadIdx.x == 0) {
      o.num_states[u] = 0, o.num_arcs[u] = 0;
      if (status >= 2) o.lattice_status[u] = 0;
    }
    return;
  }
  Lat L;
  carve_lat(L, g.ws + C.lat_off, C.NT, C.NL, g.cap, g.cap2, C.T);
  const int T = (int)C.T, nt = L.f_tok[T + 1], nl = L.f_lnk[T + 1];
  const double tot = g.tot_cost[u], beam = (double)g.lattice_beam;
  for (int i = threadIdx.x; i < nt; i += kThreads) L.extra[i] = kKeyInf, L.e_first[i] = -1, L.x_first[i] = -1;
  __syncthreads();
  for (int i = L.f_tok[T] + threadIdx.x; i < nt; i += kThreads) {  // the last frame: extra cost of ending there
    const float f = __ldg(g.finals + L.state[i]);
    const double e = status == 0 ? (f < INFINITY ? (L.alpha[i] + (double)f) - tot : INFINITY) : L.alpha[i] - tot;
    if (e <= beam) L.extra[i] = key_of(e);
  }
  __syncthreads();
  auto visit = [&](int i, const int4 k) {
    const double dx = cost_of(L.extra[k.y]);
    int keep = 0;
    if (dx < INFINITY) {
      double c = L.alpha[k.x] + (double)__ldg(g.weight + (k.z & 0x7fffffff));
      if (k.z >= 0) c += (double)__int_as_float(k.w);
      const double e = dx + (c - L.alpha[k.y]);
      if (e <= beam) keep = 1, atomicMin(L.extra + k.x, key_of(e));
    }
    L.keep[i] = keep;
  };
  for (int f = T; f >= 0; f--) {  // frames from the last, each frame's epsilon levels from the highest
    if (f < T) {
      for (int i = L.f_lnk[f + 1] + threadIdx.x; i < L.f_lnk[f + 2]; i += kThreads) {
        const int4 k = L.link[i];
        if (k.z >= 0) visit(i, k);
      }
      __syncthreads();
    }
    for (int l = g.n_lvls - 1; l >= 0; l--) {
      for (int i = L.f_lnk[f] + threadIdx.x; i < L.f_lnk[f + 1]; i += kThreads) {
        const int4 k = L.link[i];
        if (k.z < 0 && __ldg(g.lvl + L.state[k.x]) == l) visit(i, k);
      }
      __syncthreads();
    }
  }
  // runs: the links out of one token are two runs in arc order, its emitting and its epsilon arcs
  for (int i = threadIdx.x; i < nl; i += kThreads) {
    const int4 k = L.link[i];
    if (i == 0 || L.link[i - 1].x != k.x || ((L.link[i - 1].z ^ k.z) < 0)) (k.z < 0 ? L.x_first : L.e_first)[k.x] = i;
  }
  // state numbers: per frame, the rank of (level, state) among the kept tokens
  int ns = 0;
  for (int f = 0; f <= T; f++) {
    const int a = L.f_tok[f], b = L.f_tok[f + 1];
    int nk = 0;
    for (int c = a; c < b; c += kThreads) {
      const int i = c + threadIdx.x, keep = i < b && L.extra[i] != kKeyInf;
      int total;
      const int p = a + nk + block_scan(keep, sh, &total);
      if (keep) L.key[p] = ((unsigned long long)__ldg(g.lvl + L.state[i]) << 32) | (unsigned)L.state[i], L.num[i] = p;
      nk += total;
      __syncthreads();
    }
    for (int c = 0; c < nk; c += kThreads) {
      const bool mine = c + threadIdx.x < nk;
      const unsigned long long kp = mine ? L.key[a + c + threadIdx.x] : 0;
      int r = 0;
      for (int q = 0; q < nk; q += kThreads) {
        tile[threadIdx.x] = q + threadIdx.x < nk ? L.key[a + q + threadIdx.x] : ~0ull;
        __syncthreads();
        const int m = min(kThreads, nk - q);
        for (int j = 0; j < m; j++) r += tile[j] < kp;
        __syncthreads();
      }
      if (mine) L.abase[a + c + threadIdx.x] = ns + r;
    }
    __syncthreads();
    for (int i = a + threadIdx.x; i < b; i += kThreads) {
      const int n = L.extra[i] != kKeyInf ? L.abase[L.num[i]] : -1;
      if (n >= 0) {
        L.ord[n] = i;
        if (n < g.max_states) {
          const int st = L.state[i];
          o.state_frame[(int64_t)u * g.max_states + n] = f;
          o.state_graph[(int64_t)u * g.max_states + n] = st;
          o.state_final[(int64_t)u * g.max_states + n] =
              f < T ? INFINITY : status == 0 ? __ldg(g.finals + st) : 0.0f;
        }
      }
      L.num[i] = n;  // each thread rewrites only its own tokens, whose abase entries it read
    }
    ns += nk;
    __syncthreads();
  }
  // arcs: out-degrees, their prefix sum in state order, then each token's kept links merged by arc index
  auto walk = [&](int i, bool out) {
    int e = L.e_first[i], x = L.x_first[i], pos = 0;
    const int base = out ? L.abase[i] : 0;
    for (;;) {
      const bool ve = e >= 0 && e < nl && L.link[e].x == i && L.link[e].z >= 0;
      const bool vx = x >= 0 && x < nl && L.link[x].x == i && L.link[x].z < 0;
      if (!ve && !vx) break;
      const int j = ve && (!vx || L.link[e].z < (L.link[x].z & 0x7fffffff)) ? e++ : x++;
      if (!L.keep[j]) continue;
      if (out && base + pos < g.max_arcs) {
        const int4 k = L.link[j];
        const int arc = k.z & 0x7fffffff;
        const int64_t q = (int64_t)u * g.max_arcs + base + pos;
        o.arc_src[q] = L.num[i], o.arc_dst[q] = L.num[k.y];
        o.arc_ilabel[q] = __ldg(g.ilabel + arc), o.arc_olabel[q] = __ldg(g.olabel + arc);
        o.arc_graph_cost[q] = __ldg(g.weight + arc), o.arc_ac_cost[q] = k.z < 0 ? 0.0f : __int_as_float(k.w);
      }
      pos++;
    }
    return pos;
  };
  for (int i = threadIdx.x; i < nt; i += kThreads)
    if (L.num[i] >= 0) L.abase[i] = walk(i, false);
  __syncthreads();
  int na = 0;
  for (int c = 0; c < ns; c += kThreads) {
    const int n = c + threadIdx.x, i = n < ns ? L.ord[n] : 0;
    int total;
    const int p = na + block_scan(n < ns ? L.abase[i] : 0, sh, &total);
    if (n < ns) L.abase[i] = p;
    na += total;
    __syncthreads();
  }
  for (int i = threadIdx.x; i < nt; i += kThreads)
    if (L.num[i] >= 0) walk(i, true);
  if (threadIdx.x == 0) {
    o.num_states[u] = ns, o.num_arcs[u] = na;
    o.lattice_status[u] = ns > g.max_states || na > g.max_arcs ? 2 : 0;
  }
}

// The model's column of every emitting arc (outgoing order) for this call: col_of_pdf[pdf], or pdf itself.
__global__ void decode_cols_kernel(const int32_t *__restrict__ arc_pdf, const int32_t *__restrict__ col_of_pdf,
                                   int4 *__restrict__ arcs, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int p = arc_pdf[i];
    reinterpret_cast<int *>(arcs + i)[1] = col_of_pdf ? col_of_pdf[p] : p;
  }
}

// Non-finite log-likelihoods of the model's pdfs in rows [0, T) of a caller's column-ordered matrix.
__global__ void decode_count_bad_kernel(const float *__restrict__ ll, int32_t ll_stride, int64_t T,
                                        const int32_t *__restrict__ col_of_pdf, int32_t P, unsigned long long *bad) {
  unsigned long long c = 0;
  const int64_t n = T * P;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int p = (int)(i % P);
    const float v = ll[(i / P) * ll_stride + (col_of_pdf ? col_of_pdf[p] : p)];
    c += !isfinite(v);
  }
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(bad, c);
}

bool bad_cost(float v) { return std::isnan(v) || v == -INFINITY; }

size_t align16(size_t b) { return (b + 15) & ~size_t(15); }

}  // namespace

namespace vb {

int64_t decode_ws_bytes(int32_t S, int32_t cap, int32_t cap2, int32_t n_lvls, int64_t T) {
  return (int64_t)(align16((size_t)S * 8) + 3 * align16((size_t)cap * 8) + align16((size_t)cap2 * 8) +
                   align16((size_t)S * 4) + 2 * align16((size_t)cap * 4) + align16((size_t)cap2 * 4)) +
         align16((size_t)(T * cap2 * (2 + n_lvls) * 4));
}

int64_t lattice_arena_bytes(int32_t NT, int32_t NL, int32_t cap, int32_t cap2, int64_t T) {
  return (int64_t)(3 * align16((size_t)NT * 8) + align16((size_t)NL * 16) + 6 * align16((size_t)NT * 4) +
                   align16((size_t)NL * 4) + align16((size_t)cap * 4) + align16((size_t)cap2 * 4) +
                   2 * align16((size_t)(T + 2) * 4));
}

int decoder_create(int32_t num_states, int32_t start, const float *final_cost, int64_t num_arcs, const int32_t *arc_src,
                   const int32_t *arc_dst, const int32_t *arc_ilabel, const int32_t *arc_olabel, const float *arc_weight,
                   const int32_t *tid2pdf, int32_t num_tids, int device, vbgpu_decoder_t *out) {
  VB_CHECK(out, "null argument");
  *out = nullptr;
  VB_CHECK(num_states >= 1 && num_tids >= 0, "num_states %d / num_tids %d out of range", num_states, num_tids);
  VB_CHECK(num_arcs >= 0 && num_arcs < (1ll << 31), "num_arcs %lld out of range", (long long)num_arcs);
  VB_CHECK(start >= 0 && start < num_states, "start state %d outside [0, %d)", start, num_states);
  VB_CHECK(final_cost && tid2pdf, "null graph array");
  VB_CHECK(num_arcs == 0 || (arc_src && arc_dst && arc_ilabel && arc_olabel && arc_weight), "null arc array");
  const int32_t S = num_states;
  int32_t max_pdf = -1;
  for (int32_t i = 1; i <= num_tids; i++) {
    VB_CHECK(tid2pdf[i] >= 0, "tid2pdf[%d] = %d is negative", i, tid2pdf[i]);
    max_pdf = std::max(max_pdf, tid2pdf[i]);
  }
  for (int32_t s = 0; s < S; s++) VB_CHECK(!bad_cost(final_cost[s]), "final cost of state %d is NaN or -inf", s);
  for (int64_t a = 0; a < num_arcs; a++) {
    VB_CHECK(arc_src[a] >= 0 && arc_src[a] < S && arc_dst[a] >= 0 && arc_dst[a] < S,
             "arc %lld: src %d / dst %d outside the graph's %d states", (long long)a, arc_src[a], arc_dst[a], S);
    VB_CHECK(arc_ilabel[a] >= 0 && arc_ilabel[a] <= num_tids, "arc %lld: ilabel %d outside [0, %d]", (long long)a,
             arc_ilabel[a], num_tids);
    VB_CHECK(arc_olabel[a] >= 0, "arc %lld: olabel %d is negative", (long long)a, arc_olabel[a]);
    VB_CHECK(!bad_cost(arc_weight[a]), "arc %lld: weight is NaN or -inf", (long long)a);
  }
  // outgoing arcs by source, emitting and epsilon apart, each list in arc order
  std::vector<int32_t> e_off((size_t)S + 1, 0), x_off((size_t)S + 1, 0);
  for (int64_t a = 0; a < num_arcs; a++) (arc_ilabel[a] ? e_off : x_off)[arc_src[a] + 1]++;
  for (int32_t s = 0; s < S; s++) e_off[s + 1] += e_off[s], x_off[s + 1] += x_off[s];
  std::vector<int4> e_arcs((size_t)std::max(e_off[S], 1)), x_arcs((size_t)std::max(x_off[S], 1));
  std::vector<int32_t> e_pdf((size_t)std::max(e_off[S], 1), 0);
  {
    std::vector<int32_t> pe(e_off.begin(), e_off.end() - 1), px(x_off.begin(), x_off.end() - 1);
    for (int64_t a = 0; a < num_arcs; a++) {
      int32_t wbits;
      std::memcpy(&wbits, arc_weight + a, 4);
      if (arc_ilabel[a]) {
        const int32_t k = pe[arc_src[a]]++;
        e_arcs[k] = make_int4(arc_dst[a], 0, wbits, (int32_t)a);
        e_pdf[k] = tid2pdf[arc_ilabel[a]];
      } else {
        x_arcs[px[arc_src[a]]++] = make_int4(arc_dst[a], -1, wbits, (int32_t)a);
      }
    }
  }
  // epsilon levels (Kahn): level(dst) = max over epsilon arcs of level(src) + 1
  std::vector<int32_t> level((size_t)S, 0), indeg((size_t)S, 0), queue;
  for (int64_t a = 0; a < num_arcs; a++)
    if (!arc_ilabel[a]) indeg[arc_dst[a]]++;
  queue.reserve((size_t)S);
  for (int32_t s = 0; s < S; s++)
    if (!indeg[s]) queue.push_back(s);
  for (size_t q = 0; q < queue.size(); q++) {
    const int32_t s = queue[q];
    for (int32_t k = x_off[s]; k < x_off[s + 1]; k++) {
      const int32_t d = x_arcs[k].x;
      level[d] = std::max(level[d], level[s] + 1);
      if (--indeg[d] == 0) queue.push_back(d);
    }
  }
  VB_CHECK((int32_t)queue.size() == S, "the epsilon arcs of the graph form a cycle");
  const int32_t n_lvls = *std::max_element(level.begin(), level.end());

  VB_TRY(check_device(device));
  DeviceGuard g(device);
  std::unique_ptr<vbgpu_decoder_s, decltype(&vbgpu_decoder_destroy)> h(new vbgpu_decoder_s, vbgpu_decoder_destroy);
  h->device = device;
  h->S = S;
  h->start = start;
  h->num_tids = num_tids;
  h->max_pdf = max_pdf;
  h->n_lvls = n_lvls;
  h->n_emit = e_off[S];
  VB_TRY(h->stream.create());
  VB_TRY(h->d_e_off.upload(e_off.data(), e_off.size() * 4));
  VB_TRY(h->d_x_off.upload(x_off.data(), x_off.size() * 4));
  VB_TRY(h->d_e_arcs.upload(e_arcs.data(), e_arcs.size() * 16));
  VB_TRY(h->d_x_arcs.upload(x_arcs.data(), x_arcs.size() * 16));
  VB_TRY(h->d_e_pdf.upload(e_pdf.data(), e_pdf.size() * 4));
  VB_TRY(h->d_lvl.upload(level.data(), level.size() * 4));
  VB_TRY(h->d_final.upload(final_cost, (size_t)S * 4));
  VB_TRY(h->d_tid2pdf.upload(tid2pdf, (size_t)(num_tids + 1) * 4));
  const int32_t zero = 0;
  VB_TRY(h->d_ilabel.upload(num_arcs ? arc_ilabel : &zero, (size_t)std::max<int64_t>(num_arcs, 1) * 4));
  VB_TRY(h->d_olabel.upload(num_arcs ? arc_olabel : &zero, (size_t)std::max<int64_t>(num_arcs, 1) * 4));
  VB_TRY(h->d_weight.upload(num_arcs ? (const void *)arc_weight : &zero, (size_t)std::max<int64_t>(num_arcs, 1) * 4));
  *out = h.release();
  return 0;
}

int decoder_set_cols(vbgpu_decoder_t h, const int32_t *d_col_of_pdf, cudaStream_t s) {
  if (h->n_emit == 0) return 0;
  const int64_t blocks = std::min<int64_t>((h->n_emit + 255) / 256, 148 * 8);
  decode_cols_kernel<<<(unsigned)blocks, 256, 0, s>>>(h->d_e_pdf.as<int32_t>(), d_col_of_pdf, h->d_e_arcs.as<int4>(),
                                                      h->n_emit);
  VB_CUDA(cudaGetLastError());
  return 0;
}

int decoder_count_bad(const float *d_ll, int32_t ll_stride, int64_t T, const int32_t *d_col_of_pdf, int32_t P,
                      unsigned long long *bad, cudaStream_t s) {
  if (T == 0 || P == 0) return 0;
  const int64_t blocks = std::min<int64_t>((T * P + 255) / 256, 148 * 8);
  decode_count_bad_kernel<<<(unsigned)blocks, 256, 0, s>>>(d_ll, ll_stride, T, d_col_of_pdf, P, bad);
  VB_CUDA(cudaGetLastError());
  return 0;
}

int decoder_search_launch(const DecodeArgs &a, int32_t u0, int32_t n, bool lattice, cudaStream_t s) {
  if (n == 0) return 0;
  if (lattice) decode_search_kernel<true><<<n, kThreads, 0, s>>>(a, u0);
  else decode_search_kernel<false><<<n, kThreads, 0, s>>>(a, u0);
  VB_CUDA(cudaGetLastError());
  return 0;
}

int decoder_lattice_launch(const DecodeArgs &a, int32_t u0, int32_t n, cudaStream_t s) {
  if (n == 0) return 0;
  decode_lattice_kernel<<<n, kThreads, 0, s>>>(a, u0);
  VB_CUDA(cudaGetLastError());
  return 0;
}

int decoder_traceback_launch(vbgpu_decoder_t h, const DecodeArgs &a, int32_t u0, int32_t n, cudaStream_t s) {
  if (n == 0) return 0;
  decode_traceback_kernel<<<(n + 63) / 64, 64, 0, s>>>(a, u0, n, h->d_ilabel.as<int32_t>(), h->d_olabel.as<int32_t>(),
                                                       h->d_tid2pdf.as<int32_t>());
  VB_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace vb
