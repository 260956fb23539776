// score_tc.cu — dense Gaussian scoring on the sm_100a tensor cores (tcgen05.mma, accumulators in TMEM) with the
// per-pdf log-sum-exp fused into the epilogue.
//
//   loglikes[t][p] = LogSumExp_{m in pdf p}( gconst_m + means_invvars_m . x_t - 0.5 inv_vars_m . x_t^2 )
//
// which DiagGmm::LogLikelihoods (gmm/diag-gmm.cc:528-562) + VectorBase::LogSumExp (matrix/kaldi-vector.cc:757-775)
// compute per (frame, pdf) behind DecodableAmDiagGmmUnmapped::LogLikelihoodZeroBased (gmm/decodable-am-diag-gmm.cc:28-72).
// Here it is ONE contraction  Y[T x N] = A[T x K] . B[K x N]  with  K = 2D+2:
//     A row t    = [ x_0 s1_0, x_0^2 s2_0, x_1 s1_1, x_1^2 s2_1, ..., 1, 1 ]              (x already centred, see below)
//     B column g = [ miv'_0/s1_0, -0.5 iv_0/s2_0, ...,            gconst'_a, gconst'_b ] * log2(e)
// so that Y is the per-Gaussian log-likelihood in log2 units and the epilogue is exp2/log2 only.
//
// Precision.  The tensor cores take 11-bit mantissas; a single pass is ~0.05 abs off (SURVEY.md §7).  Both operands are
// therefore split in two fp16 halves (v = hi + lo, 22 bits) and three products are accumulated in the FP32 TMEM tile:
// lo.hi + hi.lo + hi.hi (lo.lo is below 2^-22 relative).  fp16 has the mantissa of TF32 at twice the MMA rate; its
// narrow exponent range is handled by exact power-of-two scales per dimension (s1, s2, chosen from the model) and by
// centring the features on the mean of the model means (c; folded exactly into miv' = miv - iv c and
// gconst' = gconst + miv.c - 0.5 iv.c^2, computed in double; gconst' is carried in three fp16 pieces over the two
// constant-one columns of A).
//
// Layout of the Gaussians (round 2).  The epilogue is the co-bottleneck of this kernel (one MUFU.EX2 per frame and
// Gaussian), so the columns are laid out for IT, not in model order:
//   * pdfs are sorted by size and taken 16 at a time into a GROUP: 16 slots x S rows, slot j / row m at column
//     m*16 + j of the group, every member padded to S Gaussians with dummy columns (score -40000).  The four epilogue
//     warps of a TMEM lane quarter own four adjacent slots each: S tcgen05.ld.x4 loads bring a warp exactly its
//     4 x S values, the log-sum-exp over the rows is straight-line code with compile-time S, and the four results of a
//     frame are one 16-byte store.  No part tables, no carries, no per-pdf branches.
//   * pdfs with 11..20 / 21..40 Gaussians span 2 / 4 adjacent slots (W = 2, 4: 8 / 4 pdfs per group); larger ones are
//     cut into virtual pdfs of <= 40 whose partial results a small merge kernel combines afterwards.
//   * a PANEL (one UMMA N, one TMA bulk copy per CTA) is a set of groups bin-packed to N = sum 16*S <= Nmax columns.
// The output therefore comes out in DEVICE COLUMN ORDER: column col_of_pdf[p] of the matrix holds pdf p (n_cols >= P
// columns: padding members and the extra pieces of cut pdfs take columns too).  Consumers index through that map — a
// decodable already goes through tid2pdf — and score_tc_launch() offers the model's pdf order through a staged gather
// kernel (row -> shared memory -> coalesced stores in pdf order).
//
// Kernel shape (persistent, warp-specialised), two variants of one template:
//   PAIR (default): CTA pairs, tcgen05.mma.cta_group::2, M = 256 frames over two SMs.  Each CTA holds the A panel of ITS
//       128 frames and HALF of every B panel (N/2 columns), so the shared-memory operand traffic per SM is half of the
//       single-CTA form (which is shared-memory-bound below N = 192) and the smem saved buys a 4-stage B ring and
//       N up to 256.  The leader CTA's MMA warp issues for both; commits are multicast to both CTAs' barriers; the
//       peer's barrier arrivals (A ready, accumulator drained, B half landed) go to the leader over DSMEM.
//   SINGLE (VBGPU_TC_SINGLE=1, and the fallback shape): one CTA per SM, two 128-frame tiles that share every B panel.
//   warp 16    producer : cp.async.bulk (TMA engine, 1-D) of the CTA's part of each B panel into a shared-memory ring.
//   warp 17    MMA      : one thread issues tcgen05.mma kind::f16 (K=16 per instruction, 3*K/16 per accumulator);
//                         accumulators live in a CIRCULAR allocation of the 512 TMEM columns (N columns per tile).
//   warp 18    relay    : (pair, peer CTA) forwards "my half of the B panel has landed" to the leader's barrier.
//   warps 0-15 epilogue : build the fp16 hi/lo A panel of the CTA's frames once per work unit (straight from the FP32
//                         features), then per accumulator: tcgen05.ld the warp's slots, hand the TMEM columns back as
//                         soon as the values are in registers, log-sum-exp, store.
// Work unit = (256-frame tile, range of B panels).  Large batches use one range (all panels); small batches and the
// tiles of the last partial wave split the panels over CTAs (pairs) to fill the GPU.
//
// The epilogue reads one precomputed entry per group from the table of its column class (dispatch key, TMEM column,
// output column); the persistent grid is sized to the CTA pairs the device keeps resident.
//
// Frames the tensor-core path cannot score are re-scored in FP32 afterwards (fix_list_kernel + fix_rows_kernel: flags ->
// list -> (frame, 32-pdf block) items over the whole grid), so they get the reference's finite answer instead of an error:
//   * features outside the fp16 plan (|x - c| beyond ~32x the model's radius), flagged while the A panel is built;
//   * frames with a result below kSunk (-27000 nats), flagged by the epilogue: that close to the dummy score of the padding
//     columns (kDummy = -40000 log2 units) the padding would show through a pdf's log-sum-exp.  Slots without a pdf score 0.
// score_tc_rescored() reports how many frames of the last launch took that path.
#include <cuda_fp16.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdlib>

#include "common.h"

namespace {

constexpr int kRowsMt = 128;   // frames per accumulator tile (TMEM lanes)
constexpr int kEpiWarps = 16;  // 4 per TMEM lane quarter
constexpr int kSmax = 10;      // rows of a group (Gaussians per slot)
constexpr int kChunkMax = 4 * kSmax;   // largest (virtual) pdf
constexpr int kAccRing = 8;    // accumulator barrier pairs (at most 6 accumulators are in flight)
constexpr int kMaxStages = 4;
constexpr float kLn2 = 0.6931471805599453f;
constexpr float kDummy = -40000.0f;    // log2-domain score of padding columns / zero-weight Gaussians
constexpr float kSunk = -27000.0f;     // nats: a result below this is within reach of the padding (kDummy ln 2 = -27726);
                                       // the frame is re-scored in FP32
constexpr double kGcMax = 4096.0;      // |gconst'| (log2 units) beyond which FP32 accumulation cannot hold 1e-3

constexpr int nmax_of(int KS, bool pair) { return pair ? 256 : 160; }
constexpr int stages_of(int KS, bool pair) { return pair ? (KS <= 5 ? 4 : 3) : 2; }

template <int KS, bool kPair>
struct Cfg {  // KS = 16-wide K steps per split; K = 16*KS >= 2D+2
  static constexpr int kc_half = 2 * KS;       // 16-byte K chunks per split
  static constexpr int kc = 4 * KS;            // hi + lo
  static constexpr int mt = kPair ? 1 : 2;     // frame tiles per CTA
  static constexpr int nmax = nmax_of(KS, kPair);
  static constexpr int stages = stages_of(KS, kPair);
  static constexpr int threads = (kEpiWarps + (kPair ? 3 : 2)) * 32;
  static constexpr int a_bytes = kc * 2048;    // one 128-row A panel: [kc][16 row groups][8 rows x 16 B]
  static constexpr int b_stage = kc * 16 * (kPair ? nmax / 2 : nmax);  // the CTA's part of the largest B panel
  static constexpr int off_b = mt * a_bytes;
  static constexpr int off_bar = off_b + stages * b_stage;
  static constexpr int smem_bytes = off_bar + 512;
};

// Panel header (int4):  x = byte offset of the panel in the image / 16 (pair: the second half follows the first),
//                       y = N | number of groups << 16,  z = index of the first group,  w = unused.
// Group entry (int2):   x = S | W << 8 | first column of the group inside the panel << 16,  y = first output column.
struct TcParams {
  const float *feats;
  int64_t T;
  int32_t stride, D;
  const uint8_t *bimg;
  const int4 *hdr;
  const int2 *grp;      // [4 column classes][grp_stride]: {dispatch key | TMEM column offset << 16, output column}
  int32_t grp_stride;
  const float *centre, *s1, *s2;  // [D]
  int32_t n_panels, n_splits;
  int64_t n_units, n_whole;
  float *out;
  int32_t ll_stride, vec_ok;
  unsigned long long *bad;
  uint8_t *rowflag;  // [T]: 1 = re-score this frame in FP32 (outside the fp16 plan)
  uint32_t dbg;      // bring-up only (VBGPU_TC_DEBUG): bit 0 = the epilogue skips loads, math and stores,
                     // bit 1 = no MMAs are issued, bit 3 = no global stores
};

// ---- PTX helpers ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Bounded wait: a protocol bug must end in a trap (a CUDA error the host reports), never in a hung GPU.  The
// suspend-time hint lets the hardware park the thread instead of re-issuing the poll (polling warps share their
// sub-partition's issue slots with the epilogue).
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  for (uint32_t spin = 0; !done; spin++) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity), "r"(20000u)
        : "memory");
    if (!done && spin > (1u << 20)) __trap();
  }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2f(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// ---- TMEM -> registers: N consecutive accumulator columns of this thread's lane (32x32b shape: lane = frame) -------------
__device__ __forceinline__ void tmem_ld1(uint32_t t, float *v) {
  uint32_t r0;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r0) : "r"(t) : "memory");
  v[0] = __uint_as_float(r0);
}
__device__ __forceinline__ void tmem_ld2(uint32_t t, float *v) {
  uint32_t r0, r1;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(t) : "memory");
  v[0] = __uint_as_float(r0), v[1] = __uint_as_float(r1);
}
__device__ __forceinline__ void tmem_ld4(uint32_t t, float *v) {
  uint32_t r[4];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(t)
               : "memory");
#pragma unroll
  for (int i = 0; i < 4; i++) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld8(uint32_t t, float *v) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(t)
               : "memory");
#pragma unroll
  for (int i = 0; i < 8; i++) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16(uint32_t t, float *v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(t)
      : "memory");
#pragma unroll
  for (int i = 0; i < 16; i++) v[i] = __uint_as_float(r[i]);
}

// ---- cluster (CTA pair) helpers ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t saddr, uint32_t rank) {  // shared::cta address -> shared::cluster
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// Wait on a barrier other CTAs of the cluster arrive on (acquire at cluster scope).
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  for (uint32_t spin = 0; !done; spin++) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity), "r"(20000u)
        : "memory");
    if (!done && spin > (1u << 20)) __trap();
  }
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint32_t bar) {  // the barrier at this offset in BOTH CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void tc_mma_f16_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ float max3f(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));  // FMNMX3
  return r;
}

// ---- one group: 16 slots x S rows of one accumulator; this warp owns slots 4*cls .. 4*cls+3 ----------------------------
// taddr = TMEM address of (the thread's lane, row 0, slot 4*cls).  S loads of four adjacent columns bring exactly the warp's
// values; as soon as they are in registers the warp may hand the TMEM columns back (rel_mode != 0: this was the warp's last
// group of the accumulator; 1 = arrive on a barrier of this CTA, 2 = on the leader CTA's over DSMEM), BEFORE the
// arithmetic — the MMA warp then only ever waits for loads, not for exponentials.
// W = slots per pdf: res[] receives 4 / W log-likelihoods (natural log).
template <int S, int W>
__device__ __forceinline__ void group_lse(uint32_t taddr, uint32_t rel_bar, uint32_t rel_mode, int lane, float (&res)[4 / W]) {
  float v[S][4];
#pragma unroll
  for (int m = 0; m < S; m++) tmem_ld4(taddr + 16u * m, v[m]);
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
  // branch-free hand-back: fence + warp sync on every group, a predicated arrive
  tc_fence_before();
  __syncwarp();
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.eq.u32 p, %1, 1;\n\t"
      "setp.eq.u32 q, %1, 2;\n\t"
      "@p mbarrier.arrive.shared::cta.b64 _, [%0];\n\t"
      "@q mbarrier.arrive.shared::cluster.b64 _, [%0];\n\t}" ::"r"(rel_bar),
      "r"(lane == 0 ? rel_mode : 0u)
      : "memory");
#pragma unroll
  for (int m = 0; m < S; m++)
#pragma unroll
    for (int j = 0; j < 4; j++) asm volatile("" : "+f"(v[m][j]));  // pin every consumer behind the wait
  if constexpr (S == 1 && W == 1) {
#pragma unroll
    for (int j = 0; j < 4; j++) res[j] = v[0][j] * kLn2;
    return;
  }
  // per-slot maxima (FMNMX3: two new values per instruction)
  float M[4];
#pragma unroll
  for (int j = 0; j < 4; j++) {
    float mx = v[0][j];
#pragma unroll
    for (int m = 1; m + 1 < S; m += 2) mx = max3f(mx, v[m][j], v[m + 1][j]);
    if constexpr ((S & 1) == 0) mx = fmaxf(mx, v[S - 1][j]);
    M[j] = mx;
  }
  if constexpr (W == 2) {
    M[0] = M[1] = fmaxf(M[0], M[1]);
    M[2] = M[3] = fmaxf(M[2], M[3]);
  } else if constexpr (W == 4) {
    M[0] = M[1] = M[2] = M[3] = max3f(fmaxf(M[0], M[1]), M[2], M[3]);
  }
  // sums of 2^(v - M): subtraction and summation as packed FP32 pairs over adjacent slots, one MUFU.EX2 per value
  const float2 nm01 = make_float2(-M[0], -M[1]), nm23 = make_float2(-M[2], -M[3]);
  float2 s01, s23;
#pragma unroll
  for (int m = 0; m < S; m++) {
    const float2 d01 = __fadd2_rn(make_float2(v[m][0], v[m][1]), nm01);
    const float2 d23 = __fadd2_rn(make_float2(v[m][2], v[m][3]), nm23);
    const float2 e01 = make_float2(ex2f(d01.x), ex2f(d01.y));
    const float2 e23 = make_float2(ex2f(d23.x), ex2f(d23.y));
    s01 = (m == 0) ? e01 : __fadd2_rn(s01, e01);
    s23 = (m == 0) ? e23 : __fadd2_rn(s23, e23);
  }
  if constexpr (W == 1) {
    res[0] = (M[0] + lg2f(s01.x)) * kLn2;
    res[1] = (M[1] + lg2f(s01.y)) * kLn2;
    res[2] = (M[2] + lg2f(s23.x)) * kLn2;
    res[3] = (M[3] + lg2f(s23.y)) * kLn2;
  } else if constexpr (W == 2) {
    res[0] = (M[0] + lg2f(s01.x + s01.y)) * kLn2;
    res[1] = (M[2] + lg2f(s23.x + s23.y)) * kLn2;
  } else {
    res[0] = (M[0] + lg2f((s01.x + s01.y) + (s23.x + s23.y))) * kLn2;
  }
}

// One group for this warp: dispatch on (S, W), store the 4 / W results of the thread's frame.
// o = &out[frame][first output column of the group + cls * 4 / W].
template <int S, int W>
__device__ __forceinline__ void run_group(uint32_t taddr, uint32_t rel_bar, uint32_t rel_mode, int lane, float *o, bool live,
                                          bool vec, float &low) {
  float res[4 / W];
  group_lse<S, W>(taddr, rel_bar, rel_mode, lane, res);
  if constexpr (W == 1) low = fminf(fminf(low, fminf(res[0], res[1])), fminf(res[2], res[3]));
  else if constexpr (W == 2) low = fminf(low, fminf(res[0], res[1]));
  else low = fminf(low, res[0]);
  if (live) {
    if constexpr (W == 1) {
      if (vec) {
        *reinterpret_cast<float4 *>(o) = make_float4(res[0], res[1], res[2], res[3]);
      } else {
        o[0] = res[0], o[1] = res[1], o[2] = res[2], o[3] = res[3];
      }
    } else if constexpr (W == 2) {
      if (vec) {
        *reinterpret_cast<float2 *>(o) = make_float2(res[0], res[1]);
      } else {
        o[0] = res[0], o[1] = res[1];
      }
    } else {
      o[0] = res[0];
    }
  }
}

// Shared-memory matrix descriptor, K-major, no swizzle (canonical layout ((8,m),(T,2)):((1T,SBO),(1,LBO))):
// a core matrix is 8 rows x 16 bytes stored contiguously (128 B); LBO = byte distance between the two core matrices
// of one K=16 step, SBO = byte distance between 8-row groups.  Bits: [0,14) addr>>4, [16,30) LBO>>4, [32,46) SBO>>4,
// [46,48) version = 1 (sm_100), [61,64) layout = 0 (no swizzle).
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) |
         (1ull << 46);
}
// Instruction descriptor for kind::f16: D = F32 (bit 4), A = B = F16 (0), both K-major (0), N>>3 at [17,23), M>>4 at [24,29).
__device__ __forceinline__ uint32_t make_idesc(uint32_t m, uint32_t n) {
  return (1u << 4) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

struct UnitRange {
  int64_t mtile;
  int32_t t0, t1;
};
// Units 0 .. n_whole-1 are whole frame tiles (all panels); the frame tiles after them are each cut into n_splits units by
// panel range.  Large batches: whole tiles fill the full waves and only the tiles of the last, partial wave are cut, so that
// the tail keeps every SM busy.  Small batches: n_whole = 0, every tile is cut.
__device__ __forceinline__ UnitRange unit_range(const TcParams &p, int64_t u) {
  UnitRange r;
  if (u < p.n_whole) {
    r.mtile = u;
    r.t0 = 0;
    r.t1 = p.n_panels;
    return r;
  }
  u -= p.n_whole;
  r.mtile = p.n_whole + u / p.n_splits;
  const int split = (int)(u - (r.mtile - p.n_whole) * p.n_splits);
  r.t0 = (int)(((int64_t)split * p.n_panels) / p.n_splits);
  r.t1 = (int)(((int64_t)(split + 1) * p.n_panels) / p.n_splits);
  return r;
}

// The accumulators take N columns each out of the 512 TMEM columns, allocated circularly in issue order (a tile that does
// not fit before column 512 starts again at 0).  Every role derives the same sequence from the panel widths alone.
struct TmemRing {
  uint32_t head = 0;
  __device__ __forceinline__ uint32_t alloc(uint32_t n) {
    if (head + n > 512u) head = 0;
    const uint32_t c = head;
    head += n;
    return c;
  }
};

// barrier slots (8 bytes each)
enum {
  kBarFull = 0,                          // [stages]   my part of the B panel has landed (TMA complete_tx)
  kBarEmpty = kBarFull + kMaxStages,     // [stages]   the MMAs that read the stage are done (tcgen05.commit)
  kBarPeerFull = kBarEmpty + kMaxStages, // [stages]   pair, leader: the peer's half has landed (relay warp, DSMEM)
  kBarAccFull = kBarPeerFull + kMaxStages,  // [kAccRing] accumulator complete (tcgen05.commit)
  kBarAccEmpty = kBarAccFull + kAccRing,    // [kAccRing] accumulator read by every epilogue warp (of both CTAs)
  kBarAReady = kBarAccEmpty + kAccRing,     // A panel(s) of the unit built
  kNumBars
};
static_assert(kNumBars * 8 <= 256, "barrier block");

template <int KS, bool kPair>
__global__ void __launch_bounds__(Cfg<KS, kPair>::threads, 1) score_tc_kernel(const TcParams p) {
  using C = Cfg<KS, kPair>;
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // tells the compiler it is warp-uniform
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + C::off_bar);
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * i; };
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + C::off_bar + 256);
  uint32_t *ring_tab = reinterpret_cast<uint32_t *>(smem + C::off_bar + 288);  // [kAccRing] column | width << 16 (MMA warp)
  uint32_t dbg;
  asm volatile("mov.u32 %0, %1;" : "=r"(dbg) : "r"(p.dbg));
  const uint32_t rank = kPair ? cluster_ctarank() : 0u;
  const bool leader = rank == 0;
  constexpr uint32_t kEpiArrivals = kPair ? 2 * kEpiWarps : kEpiWarps;
  // units are dealt to CTAs (single) or CTA pairs (pair): both CTAs of a pair walk the same sequence
  const int64_t unit0 = kPair ? (blockIdx.x >> 1) : blockIdx.x, unit_step = kPair ? (gridDim.x >> 1) : gridDim.x;

  if (threadIdx.x == kEpiWarps * 32) {
    for (int i = 0; i < C::stages; i++) {
      mbar_init(BAR(kBarFull + i), 1);
      mbar_init(BAR(kBarEmpty + i), 1);
      mbar_init(BAR(kBarPeerFull + i), 1);
    }
    for (int i = 0; i < kAccRing; i++) {
      mbar_init(BAR(kBarAccFull + i), 1);
      mbar_init(BAR(kBarAccEmpty + i), kEpiArrivals);
    }
    mbar_init(BAR(kBarAReady), kEpiArrivals);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kEpiWarps + 1) {  // TMEM: all 512 columns (one CTA per SM: the kernel takes > 180 KB of shared memory)
    if constexpr (kPair) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  if constexpr (kPair) cluster_sync_all();  // the peer's barriers are initialised before anything arrives on them
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(tmem_slot);

  if (warp == kEpiWarps) {
    // ================================================= producer =================================================
    if (lane == 0) {
      uint32_t it = 0;
      for (int64_t u = unit0; u < p.n_units; u += unit_step) {
        const UnitRange ur = unit_range(p, u);
        int4 hn = __ldg(p.hdr + ur.t0);
        for (int t = ur.t0; t < ur.t1; t++, it++) {
          const int4 h = hn;
          if (t + 1 < ur.t1) hn = __ldg(p.hdr + t + 1);
          const uint32_t s = it % C::stages, ph = (it / C::stages) & 1;
          const uint32_t n = (uint32_t)(h.y & 0xffff);
          const uint32_t bytes = (kPair ? n / 2 : n) * (uint32_t)(C::kc * 16);  // my part of the panel
          mbar_wait(BAR(kBarEmpty + s), ph ^ 1);
          mbar_expect_tx(BAR(kBarFull + s), bytes);
          bulk_g2s(smem_u32(smem + C::off_b + s * C::b_stage), p.bimg + (size_t)(uint32_t)h.x * 16 + (size_t)rank * bytes,
                   bytes, BAR(kBarFull + s));
        }
      }
    }
    __syncwarp();
  } else if (kPair && warp == kEpiWarps + 2) {
    // ================================================= relay (peer CTA of a pair) ===================================
    if (!leader && lane == 0) {
      uint32_t it = 0;
      for (int64_t u = unit0; u < p.n_units; u += unit_step) {
        const UnitRange ur = unit_range(p, u);
        for (int t = ur.t0; t < ur.t1; t++, it++) {
          const uint32_t s = it % C::stages, ph = (it / C::stages) & 1;
          mbar_wait(BAR(kBarFull + s), ph);
          mbar_arrive_remote(map_to_cta(BAR(kBarPeerFull + s), 0));
        }
      }
    }
    __syncwarp();
  } else if (warp == kEpiWarps + 1) {
    // ================================================= MMA issuer ===============================================
    // The whole warp walks the loop converged (every value below is warp-uniform, so descriptors and addresses are
    // formed in uniform registers); one elected lane issues the tensor-core instructions and the commits.  In a pair
    // only the leader CTA issues.
    if (leader) {
      uint32_t itp = 0, iti = 0, tail = 0, un = 0;
      TmemRing ring;
      const uint32_t a_base = smem_u32(smem), b_base = smem_u32(smem + C::off_b);
      for (int64_t u = unit0; u < p.n_units; u += unit_step, un++) {
        const UnitRange ur = unit_range(p, u);
        int4 hn = __ldg(p.hdr + ur.t0);
        // the A panels of this unit are in shared memory (of both CTAs)
        if constexpr (kPair) mbar_wait_cluster(BAR(kBarAReady), un & 1);
        else mbar_wait(BAR(kBarAReady), un & 1);
        for (int t = ur.t0; t < ur.t1; t++, itp++) {
          const int4 h = hn;
          if (t + 1 < ur.t1) hn = __ldg(p.hdr + t + 1);
          const uint32_t n = (uint32_t)(h.y & 0xffff);
          const uint32_t nb = kPair ? n / 2 : n;       // columns of B in this CTA's shared memory
          const uint32_t s = itp % C::stages, ph = (itp / C::stages) & 1;
          const uint32_t idesc = make_idesc(kPair ? 256u : 128u, n);
          const uint32_t kstep = 2u * nb;              // one K=16 step = two chunks of nb*16 bytes, in 16-byte units
          const uint32_t lo_off = C::kc_half * nb;     // the lo half of the panel, in 16-byte units
          mbar_wait(BAR(kBarFull + s), ph);
          if constexpr (kPair) mbar_wait(BAR(kBarPeerFull + s), ph);
          const uint64_t bdesc = make_desc(b_base + s * C::b_stage, nb * 16u, 128);
#pragma unroll 1
          for (int mt = 0; mt < C::mt; mt++, iti++) {
            // TMEM columns of this accumulator: wait for the older accumulators that still occupy them
            const uint32_t col = ring.alloc(n);
            while (tail < iti) {
              const uint32_t e = ring_tab[tail % kAccRing], ec = e & 0xffffu, en = e >> 16;
              const bool overlap = ec < col + n && col < ec + en;
              if (!overlap && iti - tail < 6u) break;
              mbar_wait(BAR(kBarAccEmpty + tail % kAccRing), (tail / kAccRing) & 1);
              tail++;
            }
            __syncwarp();
            if (lane == 0) ring_tab[iti % kAccRing] = col | (n << 16);
            __syncwarp();
            tc_fence_after();
            if (elect_one()) {
              if (!(dbg & 2u)) {
                const uint32_t d = tmem_base + col;
                const uint64_t adesc = make_desc(a_base + mt * C::a_bytes, 2048, 128);
#pragma unroll
                for (int prod = 0; prod < 3; prod++) {  // lo.hi, hi.lo, hi.hi (small terms first)
                  const uint32_t ao = (prod == 0) ? (uint32_t)(C::kc_half * 128) : 0u, bo = (prod == 1) ? lo_off : 0u;
#pragma unroll
                  for (int k = 0; k < KS; k++) {
                    if constexpr (kPair)
                      tc_mma_f16_pair(d, adesc + (ao + k * 256u), bdesc + (bo + k * kstep), idesc, (prod | k) != 0 ? 1u : 0u);
                    else
                      tc_mma_f16(d, adesc + (ao + k * 256u), bdesc + (bo + k * kstep), idesc, (prod | k) != 0 ? 1u : 0u);
                  }
                }
              }
              if constexpr (kPair) {
                tc_commit_pair(BAR(kBarAccFull + iti % kAccRing));
                tc_commit_pair(BAR(kBarEmpty + s));  // one accumulator per panel: the stage is free after these MMAs
              } else {
                tc_commit(BAR(kBarAccFull + iti % kAccRing));
                if (mt == C::mt - 1) tc_commit(BAR(kBarEmpty + s));  // the B panel (and every MMA before it) is done
              }
            }
            __syncwarp();
          }
        }
      }
    }
  } else if (warp < kEpiWarps) {
    // ================================================= epilogue =================================================
    // Warp w serves TMEM lanes 32*(w&3)..+31, i.e. frame (w&3)*32+lane of each frame tile, and slots 4*(w>>2)..+3 of
    // every group.
    const int q = warp & 3, cls = warp >> 2;
    const int2 *gcls = p.grp + (size_t)cls * p.grp_stride;  // this column class's dispatch entries
    const uint32_t tmem_q = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t iti = 0;
    TmemRing ring;
    // Non-finite results can only come from non-finite features: the model image is validated on the host, the operands
    // are bounded and every sum of exponentials is >= 1.  They are counted where the features are read.
    unsigned long long nbad = 0;
    uint32_t vec_in;  // read through an opaque move: keeps the compiler from cloning the loops per loop-invariant flag
    asm volatile("mov.u32 %0, %1;" : "=r"(vec_in) : "r"(p.vec_ok));
    const bool vec = (vec_in & 1u) != 0, no_store = (dbg & 8u) != 0;
    const uint32_t rel_mode = kPair ? 2u : 1u;
    const uint32_t aready_bar = kPair ? map_to_cta(BAR(kBarAReady), 0) : BAR(kBarAReady);
    constexpr int kRows = C::mt * kRowsMt;        // frames of this CTA per unit
    constexpr int kParts = kEpiWarps * 32 / kRows;  // threads per frame for the A build
#pragma unroll 1
    for (int64_t u = unit0; u < p.n_units; u += unit_step) {
      const UnitRange ur = unit_range(p, u);
      int4 hn = __ldg(p.hdr + ur.t0);
      const int64_t row_base = ur.mtile * 256 + (kPair ? (int64_t)rank * kRowsMt : 0);
      // ---- A panel: thread -> (row, part): K chunks part, part + kParts, ... (4 feature dims = 8 K values each) -> fp16
      //      hi/lo in the K-major core-matrix layout.  The previous unit's MMAs completed before its last accumulator was
      //      published (tcgen05.commit covers all earlier MMAs), and every epilogue warp has waited for that accumulator.
      {
        const int row = threadIdx.x % kRows, part = threadIdx.x / kRows, mt = row >> 7, rowl = row & 127;
        const int64_t trow = row_base + row;
        const float *xr = p.feats + trow * p.stride;
        bool outlier = false;
        uint8_t *arow = smem + mt * C::a_bytes + (rowl >> 3) * 128 + (rowl & 7) * 16;
#pragma unroll
        for (int i = 0; i < (2 * KS + kParts - 1) / kParts; i++) {
          const int kc = part + i * kParts;  // chunk kc: feature dims 4*kc .. 4*kc+3
          if (kc < 2 * KS) {
            float x[4] = {0.0f, 0.0f, 0.0f, 0.0f};
            if (trow < p.T) {
              if ((vec_in & 2) && 4 * kc + 3 < p.D) {  // rows are 16-byte aligned and the stride covers the padded row
                const float4 v = *reinterpret_cast<const float4 *>(xr + 4 * kc);
                x[0] = v.x, x[1] = v.y, x[2] = v.z, x[3] = v.w;
              } else {
#pragma unroll
                for (int e = 0; e < 4; e++)
                  if (4 * kc + e < p.D) x[e] = xr[4 * kc + e];
              }
            }
            __half2 hi[4], lo[4];
#pragma unroll
            for (int e = 0; e < 4; e++) {
              const int d = 4 * kc + e;  // K index 2d -> x_d * s1_d, 2d+1 -> x_d^2 * s2_d, 2D and 2D+1 -> 1
              float v0 = 0.0f, v1 = 0.0f;
              if (d < p.D) {
                const float xc = x[e] - __ldg(p.centre + d);
                v0 = xc * __ldg(p.s1 + d);
                v1 = (xc * xc) * __ldg(p.s2 + d);
                if (!(fabsf(x[e]) <= FLT_MAX)) {  // NaN / Inf feature: the reference fails on the frame's log-likelihoods
                  nbad++;
                  v0 = v1 = 0.0f;
                } else if (!(fabsf(v0) <= 65504.0f) || !(fabsf(v1) <= 65504.0f)) {  // outside the fp16 plan
                  outlier = true;
                  v0 = fminf(fmaxf(v0, -65504.0f), 65504.0f);
                  v1 = fminf(v1, 65504.0f);
                }
              } else if (d == p.D) {
                v0 = 1.0f, v1 = 1.0f;
              }
              const __half h0 = __float2half_rn(v0), h1 = __float2half_rn(v1);
              hi[e] = __halves2half2(h0, h1);
              lo[e] = __halves2half2(__float2half_rn(v0 - __half2float(h0)), __float2half_rn(v1 - __half2float(h1)));
            }
            *reinterpret_cast<uint4 *>(arow + kc * 2048) = *reinterpret_cast<uint4 *>(hi);
            *reinterpret_cast<uint4 *>(arow + (kc + C::kc_half) * 2048) = *reinterpret_cast<uint4 *>(lo);
          }
        }
        if (outlier && trow < p.T) p.rowflag[trow] = 1;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> tensor-core reads
        __syncwarp();
        if (lane == 0) {
          if constexpr (kPair) mbar_arrive_cluster(aready_bar);
          else mbar_arrive(aready_bar);
        }
      }

      // ---- panels ----
      const int64_t trow0 = row_base + q * 32 + lane;
      float low0 = 0.0f, low1 = 0.0f;
      const bool live0 = trow0 < p.T && !no_store, live1 = trow0 + kRowsMt < p.T && !no_store;
      float *orow0 = p.out + trow0 * p.ll_stride;
#pragma unroll 1
      for (int t = ur.t0; t < ur.t1; t++) {
        const int4 h = hn;
        if (t + 1 < ur.t1) hn = __ldg(p.hdr + t + 1);
        const uint32_t n = (uint32_t)(h.y & 0xffff);
        const int ng = (h.y >> 16) & 0xffff;
        const int2 *gtab = gcls + h.z;
#pragma unroll 1
        for (int mt = 0; mt < C::mt; mt++, iti++) {
          const uint32_t col = ring.alloc(n), b = iti % kAccRing, ph = (iti / kAccRing) & 1;
          float low = (mt == 0) ? low0 : low1;
          const bool live = (mt == 0) ? live0 : live1;
          float *orow = (mt == 0) ? orow0 : orow0 + (int64_t)kRowsMt * p.ll_stride;
          const uint32_t taddr = tmem_q + col;
          const uint32_t rel = kPair ? map_to_cta(BAR(kBarAccEmpty + b), 0) : BAR(kBarAccEmpty + b);
          int2 gn = __ldg(gtab);
          mbar_wait(BAR(kBarAccFull + b), ph);
          tc_fence_after();
          if (dbg & 1u) {  // bring-up: hand the columns straight back
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if constexpr (kPair) mbar_arrive_remote(rel);
              else mbar_arrive(rel);
            }
            continue;
          }
#pragma unroll 1
          for (int g = 0; g < ng; g++) {
            const int2 ge = gn;
            if (g + 1 < ng) gn = __ldg(gtab + g + 1);
            const uint32_t ta = taddr + ((uint32_t)ge.x >> 16);
            const uint32_t mode = (g + 1 == ng) ? rel_mode : 0u;
            float *o = orow + ge.y;
            switch (ge.x & 0xff) {
#define VB_CASE(S_, W_, K_) \
  case K_: run_group<S_, W_>(ta, rel, mode, lane, o, live, vec, low); break;
#define VB_CASES(W_, B_)                                                                                               \
  VB_CASE(1, W_, B_ + 0) VB_CASE(2, W_, B_ + 1) VB_CASE(3, W_, B_ + 2) VB_CASE(4, W_, B_ + 3) VB_CASE(5, W_, B_ + 4)     \
  VB_CASE(6, W_, B_ + 5) VB_CASE(7, W_, B_ + 6) VB_CASE(8, W_, B_ + 7) VB_CASE(9, W_, B_ + 8) VB_CASE(10, W_, B_ + 9)
              VB_CASES(1, 0)
              VB_CASES(2, kSmax)
              VB_CASES(4, 2 * kSmax)
#undef VB_CASES
#undef VB_CASE
              default: __trap();
            }
          }
          if (mt == 0) low0 = low;
          else low1 = low;
        }
      }
      // real scores within reach of the padding columns' dummy score: the FP32 kernel re-scores the frame
      if (low0 < kSunk && trow0 < p.T) p.rowflag[trow0] = 1;
      if (C::mt > 1 && low1 < kSunk && trow0 + kRowsMt < p.T) p.rowflag[trow0 + kRowsMt] = 1;
      __syncwarp();
    }
    if (nbad) atomicAdd(p.bad, nbad);
  }

  tc_fence_before();
  if constexpr (kPair) cluster_sync_all();  // the leader's MMAs read the peer's shared memory and write its TMEM
  else __syncthreads();
  if (warp == kEpiWarps + 1) {
    tc_fence_after();
    if constexpr (kPair)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}
static_assert(kSmax == 10, "the dispatch table above lists S = 1..10");

// ---- small companions of the tensor-core kernel -----------------------------------------------------------------------
// Frames flagged by the A-panel builder (outside the fp16 plan) or by the epilogue (scores within reach of the padding)
// are re-scored with the FP32 arithmetic of score_simt.cu (the parity anchor).  Two launches after every tensor-core
// launch: fix_list_kernel compacts the flags into a list (without flagged frames it reads T bytes and that is all), and
// fix_rows_kernel spreads (flagged frame, block of 32 pdfs) items over a persistent grid, lane = pdf.  Flagged frames
// come in runs (an utterance that went wrong), so the work must not be tied to the frame's position in the batch.
__global__ void __launch_bounds__(256) fix_list_kernel(const uint8_t *__restrict__ rowflag, int64_t T, int32_t *__restrict__ list,
                                                       unsigned int *__restrict__ count) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < T; t += (int64_t)gridDim.x * blockDim.x)
    if (rowflag[t]) list[atomicAdd(count, 1u)] = (int32_t)t;
}

__global__ void __launch_bounds__(256) fix_rows_kernel(const int32_t *__restrict__ list, const unsigned int *__restrict__ count,
                                                       const float *__restrict__ feats, int32_t stride, int32_t D, int32_t DP,
                                                       const float *__restrict__ rows, const float *__restrict__ gconsts,
                                                       const int32_t *__restrict__ pdf_offsets,
                                                       const int32_t *__restrict__ col_of_pdf, int32_t P,
                                                       float *__restrict__ out, int32_t out_stride,
                                                       unsigned long long *bad) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t nblk = (P + 31) / 32, items = (int64_t)(*count) * nblk;
  unsigned long long nbad = 0;
  for (int64_t it = warp; it < items; it += n_warps) {
    const int64_t t = list[it / nblk];
    const int pdf = (int)(it % nblk) * 32 + lane;
    if (pdf >= P) continue;
    const float *x = feats + t * stride;
    const int g0 = pdf_offsets[pdf], g1 = pdf_offsets[pdf + 1];
    float mx = -INFINITY, sum = 0.0f;
    for (int g = g0; g < g1; g++) {
      const float *row = rows + (size_t)g * 2 * DP;
      float a = 0.0f, b = 0.0f;
      for (int d = 0; d < D; d++) a = fmaf(__ldg(row + d), x[d], a);
      for (int d = 0; d < D; d++) b = fmaf(__ldg(row + DP + d), x[d] * x[d], b);
      const float ll = (__ldg(gconsts + g) + a) + b;
      if (ll > mx) {
        sum = sum * __expf(mx - ll) + 1.0f;
        mx = ll;
      } else if (ll > -INFINITY) {
        sum += __expf(ll - mx);
      }
    }
    const float res = (g1 > g0) ? mx + __logf(sum) : -INFINITY;
    if (!(fabsf(res) <= FLT_MAX)) nbad++;
    out[t * out_stride + col_of_pdf[pdf]] = res;
  }
  if (nbad) atomicAdd(bad, nbad);
}

// A pdf cut into virtual pdfs: out[t][main] = LogSumExp(out[t][main], out[t][extra_0], ...).  merge = [n][2] (main, extra),
// the entries of one pdf adjacent; a thread handles one (frame, entry run).
__global__ void __launch_bounds__(256) score_merge_kernel(float *__restrict__ out, int64_t T, int32_t out_stride,
                                                          const int32_t *__restrict__ merge, int32_t n_merge) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  float *row = out + t * out_stride;
  int i = 0;
  while (i < n_merge) {
    const int main_col = merge[2 * i];
    float mx = row[main_col], sum = 1.0f;
    for (; i < n_merge && merge[2 * i] == main_col; i++) {
      const float v = row[merge[2 * i + 1]];
      if (v > mx) {
        sum = sum * __expf(mx - v) + 1.0f;
        mx = v;
      } else {
        sum += __expf(v - mx);
      }
    }
    row[main_col] = mx + __logf(sum);
  }
}

// Device column order -> the model's pdf order: dst[t][p] = src[t][col_of_pdf[p]].
// Staged form: a persistent CTA reads a row with coalesced 16-byte loads into shared memory and writes it out in pdf order (coalesced stores, the gather happens on shared memory where
// 32 scattered words cost a few bank conflicts instead of 32 L1 wavefronts).  src is the handle's own scratch matrix
// (16-byte aligned, stride a multiple of 4).
constexpr int kGatherRows = 1;
__global__ void __launch_bounds__(256) score_gather_staged_kernel(const float *__restrict__ src, int32_t src_stride,
                                                                  const int32_t *__restrict__ col_of_pdf, int32_t P, int64_t T,
                                                                  float *__restrict__ dst, int32_t dst_stride) {
  extern __shared__ __align__(16) float gsm[];
  float *rows = gsm;  // [kGatherRows][src_stride]
  const int n4 = src_stride / 4;
  for (int64_t t0 = (int64_t)blockIdx.x * kGatherRows; t0 < T; t0 += (int64_t)gridDim.x * kGatherRows) {
    const int nr = (int)(T - t0 < kGatherRows ? T - t0 : kGatherRows);
    __syncthreads();  // the previous chunk has been written out
    const float4 *s4 = reinterpret_cast<const float4 *>(src + t0 * src_stride);
    float4 *r4 = reinterpret_cast<float4 *>(rows);
    for (int i = threadIdx.x; i < nr * n4; i += blockDim.x) r4[i] = __ldcs(s4 + i);
    __syncthreads();
    for (int r = 0; r < nr; r++) {
      float *d = dst + (t0 + r) * dst_stride;
      const float *row = rows + r * src_stride;
      for (int pdf = threadIdx.x; pdf < P; pdf += blockDim.x) __stcs(d + pdf, row[__ldg(col_of_pdf + pdf)]);
    }
  }
}
// Fallback for models whose rows do not fit in shared memory: one CTA per 8 frames, the reads gather inside a row that the
// CTA has in L1, the writes are coalesced.
__global__ void __launch_bounds__(256) score_gather_pdf_kernel(const float *__restrict__ src, int32_t src_stride,
                                                               const int32_t *__restrict__ col_of_pdf, int32_t P, int64_t T,
                                                               float *__restrict__ dst, int32_t dst_stride) {
  const int64_t t0 = (int64_t)blockIdx.x * 8;
  for (int r = 0; r < 8 && t0 + r < T; r++) {
    const float *s = src + (t0 + r) * src_stride;
    float *d = dst + (t0 + r) * dst_stride;
    for (int pdf = threadIdx.x; pdf < P; pdf += blockDim.x) d[pdf] = s[__ldg(col_of_pdf + pdf)];
  }
}

// ---- host-side state ------------------------------------------------------------------------------------------------
struct GaussPos {
  uint32_t panel;  // index into the panel tables
  uint16_t col;    // column inside the panel
};
struct TcState {
  int KS = 0, n_panels = 0, n_cols = 0, n_merge = 0, grp_stride = 0;
  bool pair = true;
  std::vector<uint8_t> h_bimg;        // kept for gconst updates
  std::vector<uint64_t> panel_off;    // byte offset of every panel in the image
  std::vector<uint16_t> panel_n;      // columns of every panel
  std::vector<GaussPos> gpos;         // where every Gaussian sits
  std::vector<double> gshift;         // gconst' - gconst  (centring term), per Gaussian
  std::vector<int32_t> col_of_pdf;    // output column of every pdf
  vb::DevBuf d_bimg, d_hdr, d_grp, d_centre, d_s1, d_s2, d_col_of_pdf, d_merge, d_rowflag, d_fixlist, d_scratch;
  bool attr_set = false, gather_attr_set = false;
  int max_pairs = 0;  // resident CTA pairs on this device (cudaOccupancyMaxActiveClusters), 0 = not asked yet
};

// Address of element (column n, K index k, half) inside a panel of N columns.  Single-CTA image: one block
// [chunk][N/8 column groups][8 columns x 16 B].  Pair image: two such blocks of N/2 columns each (what each CTA of the pair
// copies into its shared memory).  The lo half of a block follows its hi half 2*KS chunks later.
inline size_t elem_off(int N, int KS, bool pair, int n, int k, bool lo) {
  const int nb = pair ? N / 2 : N;
  const size_t block = (pair && n >= nb) ? (size_t)4 * KS * 16 * nb : 0;
  const int c = (pair && n >= nb) ? n - nb : n;
  const int chunk = k / 8 + (lo ? 2 * KS : 0);
  return block + ((size_t)chunk * (nb / 8) + c / 8) * 128 + (c % 8) * 16 + (k % 8) * 2;
}
inline void put_half(uint8_t *panel, int N, int KS, bool pair, int n, int k, bool lo, double v) {
  const __half h = __double2half(v);
  std::memcpy(panel + elem_off(N, KS, pair, n, k, lo), &h, 2);
}
inline void put_split(uint8_t *panel, int N, int KS, bool pair, int n, int k, double v) {
  const __half hi = __double2half(v);
  put_half(panel, N, KS, pair, n, k, false, v);
  put_half(panel, N, KS, pair, n, k, true, v - (double)__half2float(hi));
}
// gconst' in three fp16 pieces: hi + lo at K index 2D, the remainder at K index 2D+1 (hi half only).
inline void put_gconst(uint8_t *panel, int N, int KS, bool pair, int n, int D, double gc) {
  const __half hi = __double2half(gc);
  const double r1 = gc - (double)__half2float(hi);
  const __half lo = __double2half(r1);
  const double r2 = r1 - (double)__half2float(lo);
  put_half(panel, N, KS, pair, n, 2 * D, false, gc);
  put_half(panel, N, KS, pair, n, 2 * D, true, r1);
  put_half(panel, N, KS, pair, n, 2 * D + 1, false, r2);
  put_half(panel, N, KS, pair, n, 2 * D + 1, true, 0.0);
}

struct TcHostImage {
  std::vector<int4> hdr;
  std::vector<int2> grp;
  std::vector<int32_t> merge;
  std::vector<float> centre, s1, s2;
};

// The layout of a model for the tensor-core kernel (pure host code).  Returns null, or the reason the model is off the plan.
const char *build_layout(int D, int N, int P, const std::vector<int32_t> &po, const float *gconsts, const float *miv,
                         const float *iv, int32_t stride, bool pair, TcState *st, TcHostImage *img) {
  int KS = (2 * D + 2 + 15) / 16;
  if (KS < 2) KS = 2;
  if (KS > 6) return "feature dimension above 47";
  for (int pdf = 0; pdf < P; pdf++) {
    bool any = false;
    for (int g = po[pdf]; g < po[pdf + 1]; g++) any |= (gconsts[g] > -INFINITY);
    if (!any) return "a pdf has no Gaussian with a finite gconst";
  }
  // centre and scales from the model: means mu = miv/iv, sigma = iv^-1/2
  std::vector<double> c(D, 0.0), R(D, 0.0);
  for (int g = 0; g < N; g++)
    for (int d = 0; d < D; d++) {
      const double v = iv[(size_t)g * stride + d];
      if (!(v > 0.0) || !std::isfinite(v) || !std::isfinite((double)miv[(size_t)g * stride + d]))
        return "non-positive or non-finite variance / mean";
      c[d] += (double)miv[(size_t)g * stride + d] / v;
    }
  std::vector<float> cf(D), s1(D), s2(D);
  for (int d = 0; d < D; d++) cf[d] = (float)(c[d] / N), c[d] = (double)cf[d];
  for (int g = 0; g < N; g++)
    for (int d = 0; d < D; d++) {
      const double v = iv[(size_t)g * stride + d], mu = (double)miv[(size_t)g * stride + d] / v;
      R[d] = std::max(R[d], std::fabs(mu - c[d]) + 3.0 / std::sqrt(v));
    }
  for (int d = 0; d < D; d++) {
    const int e = (R[d] > 0.0 && std::isfinite(R[d])) ? (int)std::ceil(std::log2(R[d])) : 1000;
    if (e < -40 || e > 40) return "model radius outside the fp16 scaling plan";
    s1[d] = (float)std::ldexp(1.0, 5 - e);            // |x - c| <= R  ->  |a| <= 32
    s2[d] = (float)std::ldexp(1.0, 2 * (5 - e) - 4);  // (x - c)^2 s2 <= 64
  }

  // ---- virtual pdfs: a pdf above kChunkMax Gaussians is cut into near-equal pieces ----
  struct VPdf {
    int pdf, g0, size, piece;
  };
  std::vector<VPdf> vp;
  for (int pdf = 0; pdf < P; pdf++) {
    const int M = po[pdf + 1] - po[pdf];
    const int k = (M + kChunkMax - 1) / kChunkMax;
    int g = po[pdf];
    for (int i = 0; i < k; i++) {
      const int sz = M / k + (i < M % k ? 1 : 0);
      vp.push_back({pdf, g, sz, i});
      g += sz;
    }
  }
  // ---- groups: by slots per pdf (W = 1, 2, 4), then by size; 16 / W members per group ----
  struct Group {
    int S, W;
    std::vector<int> members;  // indices into vp
  };
  std::vector<Group> groups;
  for (int W : {1, 2, 4}) {
    std::vector<int> idx;
    for (int i = 0; i < (int)vp.size(); i++) {
      const int sz = vp[i].size, w = sz <= kSmax ? 1 : sz <= 2 * kSmax ? 2 : 4;
      if (w == W) idx.push_back(i);
    }
    std::stable_sort(idx.begin(), idx.end(), [&](int a, int b) { return vp[a].size < vp[b].size; });
    const int per = 16 / W;
    for (size_t i = 0; i < idx.size(); i += per) {
      Group gr;
      gr.W = W;
      gr.members.assign(idx.begin() + i, idx.begin() + std::min(idx.size(), i + per));
      gr.S = (vp[gr.members.back()].size + W - 1) / W;
      groups.push_back(gr);
    }
  }
  // ---- panels: groups bin-packed (first fit, tallest first) to at most nmax columns ----
  const int cap = nmax_of(KS, pair) / 16;  // rows per panel
  std::vector<int> order(groups.size());
  for (size_t i = 0; i < order.size(); i++) order[i] = (int)i;
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return groups[a].S > groups[b].S; });
  std::vector<std::vector<int>> bins;
  std::vector<int> fill;
  {
    std::vector<size_t> first_open(cap + 1, 0);  // first bin that may still take a group of S rows
    for (int gi : order) {
      const int S = groups[gi].S;
      size_t b = first_open[S];
      while (b < bins.size() && fill[b] + S > cap) b++;
      first_open[S] = b;
      if (b == bins.size()) {
        bins.emplace_back();
        fill.push_back(0);
      }
      bins[b].push_back(gi);
      fill[b] += S;
    }
  }
  st->KS = KS;
  st->pair = pair;
  st->gpos.resize(N);
  st->gshift.assign(N, 0.0);
  st->col_of_pdf.assign(P, -1);
  std::vector<int4> &hdr = img->hdr;
  std::vector<int2> &grp = img->grp;
  std::vector<int32_t> &merge = img->merge;  // (main column, extra column)
  std::vector<int32_t> vcol(vp.size(), -1);
  std::vector<int> group_col0(groups.size(), 0);
  {
    // output columns: W = 1 groups first (16 columns each), then W = 2 (8), then W = 4 (4): keeps 16-byte stores aligned
    std::vector<int> group_out(groups.size(), 0);
    int out_col = 0;
    for (int W : {1, 2, 4})
      for (size_t b = 0; b < bins.size(); b++)
        for (int gi : bins[b])
          if (groups[gi].W == W) {
            group_out[gi] = out_col;
            for (size_t j = 0; j < groups[gi].members.size(); j++) vcol[groups[gi].members[j]] = out_col + (int)j;
            out_col += 16 / W;
          }
    st->n_cols = (out_col + 3) / 4 * 4;
    uint64_t off = 0;
    for (size_t b = 0; b < bins.size(); b++) {
      const int Np = 16 * fill[b];
      st->panel_off.push_back(off);
      st->panel_n.push_back((uint16_t)Np);
      hdr.push_back(make_int4((int)(off / 16), Np | ((int)bins[b].size() << 16), (int)grp.size(), 0));
      int col0 = 0;
      for (int gi : bins[b]) {
        group_col0[gi] = col0;
        grp.push_back(make_int2(groups[gi].S | (groups[gi].W << 8) | (col0 << 16), group_out[gi]));
        col0 += 16 * groups[gi].S;
      }
      off += (uint64_t)4 * KS * 16 * Np;
    }
    st->n_panels = (int)hdr.size();
    st->h_bimg.assign(off, 0);
    hdr.push_back(make_int4(0, 16 | (1 << 16), 0, 0));  // padding entry: the kernel may prefetch one past the end
    grp.push_back(make_int2(1 | (1 << 8), 0));
  }
  for (size_t i = 0; i < vp.size(); i++)
    if (vp[i].piece == 0) st->col_of_pdf[vp[i].pdf] = vcol[i];
  for (size_t i = 0; i < vp.size(); i++)
    if (vp[i].piece > 0) {
      merge.push_back(st->col_of_pdf[vp[i].pdf]);
      merge.push_back(vcol[i]);
    }
  st->n_merge = (int)merge.size() / 2;
  // ---- B image ----
  const double L2E = 1.4426950408889634074;
  const char *why = nullptr;
  for (int pi = 0; pi < st->n_panels && !why; pi++) {
    const int Np = st->panel_n[pi];
    uint8_t *panel = st->h_bimg.data() + st->panel_off[pi];
    std::vector<int> gauss_of_col(Np, -1);
    for (int gi : bins[pi]) {
      const Group &gr = groups[gi];
      for (size_t j = 0; j < gr.members.size(); j++) {
        const VPdf &v = vp[gr.members[j]];
        for (int k = 0; k < v.size; k++) gauss_of_col[group_col0[gi] + (k / gr.W) * 16 + gr.W * (int)j + k % gr.W] = v.g0 + k;
      }
    }
    // a slot without a pdf scores 0 instead of the dummy level: the epilogue takes any result near the dummy level as a
    // frame whose real scores sank below the padding and hands the frame to the FP32 kernel
    std::vector<uint8_t> idle(Np, 0);
    for (int gi : bins[pi]) {
      const Group &gr = groups[gi];
      for (int j = (int)gr.members.size(); j < 16 / gr.W; j++) idle[group_col0[gi] + gr.W * j] = 1;
    }
    for (int n = 0; n < Np && !why; n++) {
      const int g = gauss_of_col[n];
      double gc = idle[n] ? 0.0 : (double)kDummy;
      if (g >= 0) {
        st->gpos[g] = {(uint32_t)pi, (uint16_t)n};
        double shift = 0.0;
        for (int d = 0; d < D; d++) {
          const double v = iv[(size_t)g * stride + d], mv = miv[(size_t)g * stride + d];
          const double b1 = (mv - v * c[d]) * L2E / (double)s1[d], b2 = -0.5 * v * L2E / (double)s2[d];
          if (std::fabs(b1) > 60000.0 || std::fabs(b2) > 60000.0) why = "model parameters outside the fp16 range";
          put_split(panel, Np, KS, pair, n, 2 * d, b1);
          put_split(panel, Np, KS, pair, n, 2 * d + 1, b2);
          shift += mv * c[d] - 0.5 * v * c[d] * c[d];
        }
        st->gshift[g] = shift;
        if (gconsts[g] > -INFINITY) {  // a zero-weight Gaussian keeps the dummy score
          gc = ((double)gconsts[g] + shift) * L2E;
          if (!(std::fabs(gc) <= kGcMax)) why = "a centred gconst is too large for FP32 accumulation at 1e-3";
        }
      }
      put_gconst(panel, Np, KS, pair, n, D, gc);
    }
  }
  img->centre = cf, img->s1 = s1, img->s2 = s2;
  return why;
}

template <int KS, bool kPair>
int launch_ks(const TcParams &p, TcState *st, int grid, cudaStream_t s) {
  using C = Cfg<KS, kPair>;
  if (!st->attr_set) {
    VB_CUDA(cudaFuncSetAttribute(score_tc_kernel<KS, kPair>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::smem_bytes));
    st->attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(C::threads);
  cfg.dynamicSmemBytes = C::smem_bytes;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kPair ? 2 : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  VB_CUDA(cudaLaunchKernelEx(&cfg, score_tc_kernel<KS, kPair>, p));
  return 0;
}
// How many CTA pairs of the kernel the device keeps resident at once.  A persistent grid must not be larger: on a part whose
// floor-sweeping leaves a GPC with an odd number of usable SMs fewer than SMs / 2 pairs fit, and the pairs that do not fit
// would run as a second wave, after the others have finished their share.
template <int KS>
int max_pairs_ks(int *out) {
  using C = Cfg<KS, true>;
  VB_CUDA(cudaFuncSetAttribute(score_tc_kernel<KS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::smem_bytes));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2);
  cfg.blockDim = dim3(C::threads);
  cfg.dynamicSmemBytes = C::smem_bytes;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  VB_CUDA(cudaOccupancyMaxActiveClusters(out, score_tc_kernel<KS, true>, &cfg));
  return 0;
}
int max_pairs(int KS, int *out) {
  switch (KS) {
    case 2: return max_pairs_ks<2>(out);
    case 3: return max_pairs_ks<3>(out);
    case 4: return max_pairs_ks<4>(out);
    case 5: return max_pairs_ks<5>(out);
    case 6: return max_pairs_ks<6>(out);
    default: return vb::fail(VBGPU_ERR_INVALID, "unsupported K for the tensor-core scorer");
  }
}

template <bool kPair>
int launch_any(const TcParams &p, TcState *st, int grid, cudaStream_t s) {
  switch (st->KS) {
    case 2: return launch_ks<2, kPair>(p, st, grid, s);
    case 3: return launch_ks<3, kPair>(p, st, grid, s);
    case 4: return launch_ks<4, kPair>(p, st, grid, s);
    case 5: return launch_ks<5, kPair>(p, st, grid, s);
    case 6: return launch_ks<6, kPair>(p, st, grid, s);
    default: return vb::fail(VBGPU_ERR_INVALID, "unsupported K for the tensor-core scorer");
  }
}

void note_fallback(vbgpu_gmm_t h, const char *why) {
  h->tc_note = why;
  if (!getenv("VBGPU_QUIET"))
    fprintf(stderr, "vbgpu: model (P=%d N=%d D=%d) is scored by the FP32 SIMT kernel, not tcgen05: %s\n", h->P, h->N, h->D, why);
}

}  // namespace

namespace vb {

void score_tc_release(vbgpu_gmm_t h) {
  delete static_cast<TcState *>(h->tc);
  h->tc = nullptr;
}

bool score_tc_available(vbgpu_gmm_t h) { return h->tc != nullptr; }
// Frames the last launch handed to the FP32 kernel (synchronises the device); 0 when the model is not on the plan.
int score_tc_rescored(vbgpu_gmm_t h, int64_t *n) {
  *n = 0;
  TcState *st = static_cast<TcState *>(h->tc);
  if (!st || !st->d_fixlist.p) return 0;
  VB_CUDA(cudaDeviceSynchronize());
  unsigned int v = 0;
  VB_CUDA(cudaMemcpy(&v, st->d_fixlist.p, 4, cudaMemcpyDeviceToHost));
  *n = (int64_t)v;
  return 0;
}

int32_t score_tc_num_cols(vbgpu_gmm_t h) { return h->tc ? static_cast<TcState *>(h->tc)->n_cols : h->P; }
const int32_t *score_tc_col_of_pdf(vbgpu_gmm_t h) {
  return h->tc ? static_cast<TcState *>(h->tc)->col_of_pdf.data() : nullptr;
}
const int32_t *score_tc_col_of_pdf_dev(vbgpu_gmm_t h) {
  return h->tc ? static_cast<TcState *>(h->tc)->d_col_of_pdf.as<int32_t>() : nullptr;
}

// Builds the tensor-core image of the model.  Leaves h->tc null (the SIMT kernel serves the model, h->tc_note says why)
// when the model does not fit: D > 47, a pdf with no finite gconst, or values outside the fp16 plan.
int score_tc_prepare(vbgpu_gmm_t h, const float *gconsts, const float *miv, const float *iv, int32_t stride) {
  h->tc_note = "";
  if (getenv("VBGPU_DISABLE_TC")) {
    h->tc_note = "VBGPU_DISABLE_TC is set";
    return 0;
  }
  const char *single = getenv("VBGPU_TC_SINGLE");
  const bool pair = !(single && atoi(single) != 0);
  std::unique_ptr<TcState> st(new TcState);
  TcHostImage img;
  const char *why = build_layout(h->D, h->N, h->P, h->h_pdf_offsets, gconsts, miv, iv, stride, pair, st.get(), &img);
  if (why) {
    note_fallback(h, why);
    return 0;
  }
  auto up = [](DevBuf &b, const void *src, size_t bytes) {  // every table gets at least 16 bytes
    VB_TRY(b.reserve(std::max<size_t>(bytes, 16)));
    return b.upload(src, bytes);
  };
  VB_TRY(up(st->d_bimg, st->h_bimg.data(), st->h_bimg.size()));
  VB_TRY(up(st->d_hdr, img.hdr.data(), img.hdr.size() * sizeof(int4)));
  {  // dispatch entries per column class (warp >> 2): everything the epilogue would otherwise derive per group
    const size_t ng = img.grp.size();
    std::vector<int2> dev(4 * ng);
    for (int cls = 0; cls < 4; cls++)
      for (size_t g = 0; g < ng; g++) {
        const int S = img.grp[g].x & 0xff, W = (img.grp[g].x >> 8) & 0xff, col0 = (img.grp[g].x >> 16) & 0xffff;
        const int key = (S - 1) + (W == 1 ? 0 : W == 2 ? kSmax : 2 * kSmax);
        dev[cls * ng + g] = make_int2(key | ((col0 + 4 * cls) << 16), img.grp[g].y + cls * (4 / W));
      }
    VB_TRY(up(st->d_grp, dev.data(), dev.size() * sizeof(int2)));
    st->grp_stride = (int)ng;
  }
  VB_TRY(up(st->d_centre, img.centre.data(), h->D * 4));
  VB_TRY(up(st->d_s1, img.s1.data(), h->D * 4));
  VB_TRY(up(st->d_s2, img.s2.data(), h->D * 4));
  VB_TRY(up(st->d_col_of_pdf, st->col_of_pdf.data(), (size_t)h->P * 4));
  VB_TRY(up(st->d_merge, img.merge.data(), img.merge.size() * 4));
  h->tc = st.release();
  return 0;
}

// Host-only view of the layout (no device needed): what tests/test_tc_layout.py decodes and checks against the oracle.
// info[8] = {K steps, panels, columns, merge entries, image bytes / 16, groups, pair, slots per group}.  bounds[64][65]
// (nullable) receives the panel ranges of a frame tile cut into k = 1..64 units, as unit_range() computes them.
int score_tc_debug_layout(int32_t P, int32_t D, const int32_t *pdf_offsets, const float *gconsts, const float *miv,
                          const float *iv, int32_t stride, int32_t pair, int32_t *info, uint8_t *image, int64_t image_cap,
                          int32_t *hdr, int32_t hdr_cap, int32_t *grp, int32_t grp_cap, int32_t *col_of_pdf, int32_t *merge,
                          int32_t merge_cap, float *centre, float *s1, float *s2, int32_t *bounds) {
  TcState st;
  TcHostImage img;
  std::vector<int32_t> po(pdf_offsets, pdf_offsets + P + 1);
  const char *why = build_layout(D, po[P], P, po, gconsts, miv, iv, stride, pair != 0, &st, &img);
  if (why) return fail(VBGPU_ERR_INVALID, "not on the tensor-core plan: %s", why);
  const int n_groups = (int)img.grp.size() - 1;
  info[0] = st.KS, info[1] = st.n_panels, info[2] = st.n_cols, info[3] = st.n_merge;
  info[4] = (int32_t)(st.h_bimg.size() >> 4), info[5] = n_groups, info[6] = pair != 0, info[7] = 16;
  if (image && (int64_t)st.h_bimg.size() <= image_cap) std::memcpy(image, st.h_bimg.data(), st.h_bimg.size());
  if (hdr && st.n_panels * 4 <= hdr_cap) std::memcpy(hdr, img.hdr.data(), (size_t)st.n_panels * 16);
  if (grp && n_groups * 2 <= grp_cap) std::memcpy(grp, img.grp.data(), (size_t)n_groups * 8);
  if (col_of_pdf) std::memcpy(col_of_pdf, st.col_of_pdf.data(), (size_t)P * 4);
  if (merge && (int)img.merge.size() <= merge_cap) std::memcpy(merge, img.merge.data(), img.merge.size() * 4);
  if (centre) std::memcpy(centre, img.centre.data(), D * 4);
  if (s1) std::memcpy(s1, img.s1.data(), D * 4);
  if (s2) std::memcpy(s2, img.s2.data(), D * 4);
  if (bounds)
    for (int k = 1; k <= 64; k++)
      for (int i = 0; i <= 64; i++) bounds[(k - 1) * 65 + i] = (int32_t)(((int64_t)std::min(i, k) * st.n_panels) / k);
  return 0;
}

int score_tc_update_gconsts(vbgpu_gmm_t h, const float *gconsts) {
  TcState *st = static_cast<TcState *>(h->tc);
  if (!st) return 0;
  const std::vector<int32_t> &po = h->h_pdf_offsets;
  for (int pdf = 0; pdf < h->P; pdf++) {
    bool any = false;
    for (int g = po[pdf]; g < po[pdf + 1]; g++) any |= (gconsts[g] > -INFINITY);
    if (!any) {  // a pdf without a finite gconst: only the SIMT kernel reproduces the reference's -inf
      score_tc_release(h);
      note_fallback(h, "a pdf has no Gaussian with a finite gconst");
      return 0;
    }
  }
  const double L2E = 1.4426950408889634074;
  for (int g = 0; g < h->N; g++) {
    double gc = kDummy;
    if (gconsts[g] > -INFINITY) {
      gc = ((double)gconsts[g] + st->gshift[g]) * L2E;
      if (!(std::fabs(gc) <= kGcMax)) {
        score_tc_release(h);
        note_fallback(h, "a centred gconst is too large for FP32 accumulation at 1e-3");
        return 0;
      }
    }
    const GaussPos gp = st->gpos[g];
    put_gconst(st->h_bimg.data() + st->panel_off[gp.panel], st->panel_n[gp.panel], st->KS, st->pair, gp.col, h->D, gc);
  }
  VB_CUDA(cudaMemcpy(st->d_bimg.p, st->h_bimg.data(), st->h_bimg.size(), cudaMemcpyHostToDevice));
  return 0;
}

// Scores T frames.  native != 0: d_ll is [T x ll_stride] in DEVICE COLUMN ORDER (ll_stride >= score_tc_num_cols());
// native == 0: d_ll is [T x ll_stride] in the model's pdf order (the kernel writes a scratch matrix, a gather kernel
// produces d_ll).
int score_tc_launch(vbgpu_gmm_t h, const float *d_feats, int64_t T, int32_t stride, float *d_ll, int32_t ll_stride,
                    int native, unsigned long long *bad, cudaStream_t s) {
  TcState *st = static_cast<TcState *>(h->tc);
  if (!st) return fail(VBGPU_ERR_INVALID, "tensor-core scorer unavailable for this model");
  if (T == 0) return 0;
  if (T >= (1LL << 31) - 512) return fail(VBGPU_ERR_INVALID, "too many frames in one call");
  float *out = d_ll;
  int32_t out_stride = ll_stride;
  if (!native) {
    out_stride = st->n_cols;
    VB_TRY(st->d_scratch.reserve((size_t)T * out_stride * 4));
    out = st->d_scratch.as<float>();
  } else if (ll_stride < st->n_cols) {
    return fail(VBGPU_ERR_INVALID, "ll_stride %d < %d device columns", ll_stride, st->n_cols);
  }
  VB_TRY(st->d_rowflag.reserve((size_t)T));
  VB_CUDA(cudaMemsetAsync(st->d_rowflag.p, 0, (size_t)T, s));
  VB_TRY(st->d_fixlist.reserve(16 + (size_t)T * 4));  // [count, pad][flagged frames]
  VB_CUDA(cudaMemsetAsync(st->d_fixlist.p, 0, 16, s));
  const int sms = num_sms(h->device);
  if (st->pair && st->max_pairs == 0) {
    VB_TRY(max_pairs(st->KS, &st->max_pairs));
    if (st->max_pairs < 1) return fail(VBGPU_ERR_CUDA, "the device cannot hold one CTA pair of the scoring kernel");
    if (st->max_pairs < sms / 2 && !getenv("VBGPU_QUIET"))
      fprintf(stderr, "vbgpu: device %d keeps %d CTA pairs of the scoring kernel resident (%d SMs): the grid is sized to that\n",
              h->device, st->max_pairs, sms);
  }
  // CTAs, or CTA pairs: each takes 256-frame units
  const int workers = st->pair ? std::min(sms / 2, getenv("VBGPU_TC_IGNORE_OCCUPANCY") ? sms / 2 : st->max_pairs) : sms;
  const int64_t n_mtiles = (T + 255) / 256;
  // split the panels over the workers when there are too few frame tiles: pick the split with the best last-wave fill
  int best = 1;
  int64_t n_whole = 0;
  if (n_mtiles < 4LL * workers) {
    double best_eff = 0.0;
    const int max_split = std::min(st->n_panels, 64);
    for (int k = 1; k <= max_split; k++) {
      const int64_t units = n_mtiles * k, waves = (units + workers - 1) / workers;
      // each extra split repeats the A-panel build: charge it as ~2 panels of work per unit
      const double work = (double)st->n_panels / k + 2.0;
      const double eff = ((double)st->n_panels / k) / work * (double)units / (double)(waves * workers);
      if (eff > best_eff * 1.02) best_eff = eff, best = k;
    }
  } else {
    // many tiles: whole tiles for the full waves; the r tiles of the last, partial wave are cut into floor(workers / r)
    // panel ranges each so that the tail runs on (almost) every SM for 1/k of a tile's time instead of on r of them
    const int64_t r = n_mtiles % workers;
    int k = r > 0 ? (int)std::min<int64_t>(std::min(st->n_panels, 16), workers / r) : 1;
    if (getenv("VBGPU_TC_NO_TAIL_SPLIT")) k = 1;  // bring-up: A/B of the tail split
    if (k >= 2) best = k, n_whole = n_mtiles - r;
    else n_whole = n_mtiles;
  }
  TcParams p;
  p.feats = d_feats;
  p.T = T;
  p.stride = stride;
  p.D = h->D;
  p.bimg = st->d_bimg.as<uint8_t>();
  p.hdr = st->d_hdr.as<int4>();
  p.grp = st->d_grp.as<int2>();
  p.grp_stride = st->grp_stride;
  p.centre = st->d_centre.as<float>();
  p.s1 = st->d_s1.as<float>();
  p.s2 = st->d_s2.as<float>();
  p.n_panels = st->n_panels;
  p.n_splits = best;
  p.n_whole = n_whole;
  p.n_units = n_whole + (n_mtiles - n_whole) * best;
  p.out = out;
  p.ll_stride = out_stride;
  const int padded = (h->D + 3) / 4 * 4;
  p.vec_ok = (((reinterpret_cast<uintptr_t>(out) & 15) == 0 && out_stride % 4 == 0) ? 1 : 0) |
             (((reinterpret_cast<uintptr_t>(d_feats) & 15) == 0 && stride % 4 == 0 && stride >= padded) ? 2 : 0);
  p.bad = bad;
  p.rowflag = st->d_rowflag.as<uint8_t>();
  const char *dbg_env = getenv("VBGPU_TC_DEBUG");
  p.dbg = dbg_env ? (uint32_t)atoi(dbg_env) : 0u;
  const int n_workers = (int)std::min<int64_t>(p.n_units, workers);
  VB_TRY(st->pair ? launch_any<true>(p, st, 2 * n_workers, s) : launch_any<false>(p, st, n_workers, s));
  if (st->n_merge > 0) {
    score_merge_kernel<<<(unsigned)((T + 255) / 256), 256, 0, s>>>(out, T, out_stride, st->d_merge.as<int32_t>(), st->n_merge);
    VB_CUDA(cudaGetLastError());
  }
  {
    int32_t *list = reinterpret_cast<int32_t *>(st->d_fixlist.as<uint8_t>() + 16);
    unsigned int *count = st->d_fixlist.as<unsigned int>();
    fix_list_kernel<<<(unsigned)std::min<int64_t>((T + 255) / 256, 2LL * sms), 256, 0, s>>>(st->d_rowflag.as<uint8_t>(), T, list, count);
    VB_CUDA(cudaGetLastError());
    fix_rows_kernel<<<4 * sms, 256, 0, s>>>(list, count, d_feats, stride, h->D, h->DP, h->d_rows.as<float>(),
                                            h->d_gconsts.as<float>(), h->d_pdf_offsets.as<int32_t>(),
                                            st->d_col_of_pdf.as<int32_t>(), h->P, out, out_stride, p.bad);
    VB_CUDA(cudaGetLastError());
  }
  if (!native) {
    const size_t gsm = sizeof(float) * (size_t)kGatherRows * out_stride;
    if (gsm <= 100 * 1024 && out_stride % 4 == 0) {
      if (!st->gather_attr_set) {
        VB_CUDA(cudaFuncSetAttribute(score_gather_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        st->gather_attr_set = true;
      }
      const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / std::max<size_t>(gsm, 1)));
      const unsigned blocks = (unsigned)std::min<int64_t>((T + kGatherRows - 1) / kGatherRows, (int64_t)per_sm * sms);
      score_gather_staged_kernel<<<blocks, 256, gsm, s>>>(out, out_stride, st->d_col_of_pdf.as<int32_t>(), h->P, T, d_ll,
                                                          ll_stride);
    } else {
      score_gather_pdf_kernel<<<(unsigned)((T + 7) / 8), 256, 0, s>>>(out, out_stride, st->d_col_of_pdf.as<int32_t>(), h->P, T,
                                                                     d_ll, ll_stride);
    }
    VB_CUDA(cudaGetLastError());
  }
  return 0;
}

}  // namespace vb
