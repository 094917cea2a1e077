// K1 front end on the 5th-generation tensor cores (sm_100a): fp16 tcgen05.mma with TMEM
// accumulators, operands staged by TMA, candidate tracking fused into the TMEM epilogue.
//
// Replaces the distance evaluation inside BaseSom._get_winning_neurons (dbgsom/BaseSom.py:446-464;
// the reference runs sklearn's float64 GEMM expansion ||x||^2 - 2 x.w + ||w||^2).  Here the score
// of prototype j for sample i is  s_ij = wnorm_j - 2 x'_i . u_j  with the shadows of
// dbgsom_prepare_x16 / dbgsom_prepare_w (x' centred on the data, u centred on the prototype mean,
// both scaled by a power of two; s_ij equals the squared distance up to a per-sample constant).
//   n_pass = 1 :  x'.u ~ xh.uh                          (fp16 inputs, error ~ 2^-9  ||x'|| ||u||)
//   n_pass = 3 :  x'.u ~ xh.uh + xh.ul + xl.uh          (split fp16,  error ~ 2^-20 ||x'|| ||u||)
// all products accumulate in one fp32 TMEM tile.  The epilogue never writes the N x M score
// matrix: each of its threads owns one TMEM lane = one sample row, streams the scores of all M
// prototypes through a small candidate table (gate / slow_offer below) and emits at most
// DBGSOM_MAX_CAND candidates per sample for the exact float64 re-score (bmu_resolve.cu).
//
// CTA = 128 sample rows x all prototypes, persistent over row tiles.  Warp roles:
//   warp 0      TMA producer (one elected lane)
//   warp 1      MMA issuer   (one elected lane).  Default: CTA PAIRS -- the leader CTA of a cluster of two
//               issues tcgen05.mma.cta_group::2 (M = 256: 128 rows of each CTA; N = 128 with the sample tile
//               in tensor memory for D <= 256, N = 256 with both operands streamed beyond), each CTA stages
//               half of every prototype tile.  Otherwise cta_group::1, M = 128, optionally with the
//               prototype tiles TMA-multicast to a cluster.
//   warp 2      TMEM allocate / free
//   warps 4-19  epilogue: tcgen05.ld 32x32b -> registers -> score -> candidate tracking.
//               A warp can only read the 32 TMEM lanes of its scheduler quarter (warp % 4), so four
//               warps share each quarter and take every fourth 32-column chunk: one warp per
//               scheduler runs at IPC ~0.06 (measured), four hide each other's latencies.  The four
//               trackers of a row share their running minimum through shared memory and are merged
//               at the end of the row tile.
// Prototypes are visited in a fixed scattered order (the shadow rows are permuted by
// dbgsom_prepare_w; shadow row c holds prototype (c * stride) % Mpad): in map order a smooth map makes
// the scores fall monotonically towards the best region, so nearly every chunk would set a new
// running minimum; in scattered order only ~ln(#chunks) do.
// Pipelines: smem ring full/empty (TMA <-> MMA), TMEM double buffer full/empty (MMA <-> epilogue),
// and, when the whole K extent of the sample tile fits (XRES), a resident A tile loaded once per
// row tile so that only prototypes stream from L2.
#include <cuda.h>

#include <cstdio>
#include <cstdlib>

#include "common.cuh"

namespace dbgsom {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;  // fp16 elements = one 128-byte swizzle atom row
constexpr int UMMA_K = 16;
constexpr int A_TILE_BYTES = BM * BK * 2;  // 16 KB
constexpr int EPI_WARP0 = 4;
constexpr int EPI_SUBS = 4;   // epilogue warps per TMEM lane quarter
constexpr int EPI_WARPS = 4 * EPI_SUBS;
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int TC_THREADS = (EPI_WARP0 + EPI_WARPS) * 32;  // 640
constexpr int KSUB = 4;       // candidate slots per (row, epilogue warp)
constexpr int MAX_RES_KB = 4;  // resident A up to D = 256
constexpr int kFlagMaxCols = 4096;                         // selective search: prototypes (padded) it covers
constexpr int kFlagChunkBytes = kFlagMaxCols / 32 * BM * 4;  // FLAG pass: float minimum per (32-column chunk, row)
// top-k search (NB > 2): per (row, epilogue warp) a sorted table of up to KTOP (score, prototype) pairs, laid out
// [sub][slot][row] so that the 32 rows of a warp hit 32 banks; values, then indices
constexpr int KTOP = kMaxNbmu;
constexpr uint32_t kTopIdxOffset = EPI_SUBS * KTOP * BM * 4;
constexpr int kTopTabBytes = 2 * EPI_SUBS * KTOP * BM * 4;  // 64 KB, taken from the operand ring
template <int NB, int SEL>
__host__ __device__ constexpr int extra_bytes() { return SEL == 1 ? kFlagChunkBytes : (NB > 2 ? kTopTabBytes : 0); }

// ------------------------------------------------------------------------------------------ PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// try_wait suspends the thread in hardware up to the time hint (ns) instead of spinning, so the
// single-lane producer / MMA warps do not steal issue slots from the epilogue warp of their SMSP.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity), "r"(20000u)
      : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(x), "r"(y)
      : "memory");
}
// same, delivered to the same shared-memory offset (and signalled on the same barrier offset) in every CTA of
// the cluster named in cta_mask: one L2 read feeds all of them
__device__ __forceinline__ void tma_load_2d_mc(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int x, int y,
                                               uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, "
      "{%3, %4}], [%2], %5;" ::"r"(smem_u32(smem_dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(x), "r"(y), "h"(cta_mask)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// arrive on the barrier at this offset in every CTA of cta_mask once the MMAs issued so far have completed
__device__ __forceinline__ void tc_commit_mc(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}
// D[tmem] (+)= A[smem] . B[smem]^T, fp16 inputs, fp32 accumulate
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same with the A operand read from tensor memory (128 lanes = rows, 2 fp16 per 32-bit column)
__device__ __forceinline__ void tc_mma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// shared memory -> tensor memory: 128 rows x 256 bit (one K = 16 slice of an fp16 operand tile)
__device__ __forceinline__ void tc_cp_128x256b(uint32_t tmem_dst, uint64_t desc_src) {
  asm volatile("tcgen05.cp.cta_group::1.128x256b [%0], %1;" ::"r"(tmem_dst), "l"(desc_src) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- CTA pair (cta_group::2): one MMA stream for two SMs.  The leader CTA (cluster rank 0) issues every
// tcgen05.mma / tcgen05.cp / tcgen05.commit for both; each CTA keeps its own sample rows in its own tensor
// memory and holds HALF of every prototype tile in its own shared memory (the pair exchanges the halves inside
// the TPC), so shared-memory reads and TMA writes per SM are half of the single-CTA form.
__device__ __forceinline__ uint32_t mapa_u32(uint32_t cta_addr, uint32_t rank) {  // shared::cluster address in `rank`
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(cta_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  // default semantics (release at CTA scope), like CUTLASS' ClusterBarrier::arrive(cta_id): the data this barrier
  // guards moves through the async / tensor proxies, whose ordering comes from complete_tx and the tcgen05 fences;
  // `.release.cluster` put a full error-barrier fence (~300 cycles) in front of every arrive
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load into MY shared memory, completion bytes counted on the barrier at `bar_cluster_addr` (the leader's)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int x,
                                                 int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
          "r"(smem_u32(smem_dst)),
      "l"(map), "r"(bar_cluster_addr), "r"(x), "r"(y)
      : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}
__device__ __forceinline__ void tc_mma_f16_ts_pair(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                                   uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same with the A operand from shared memory (each CTA's own tile at the same offset)
__device__ __forceinline__ void tc_mma_f16_ss_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                   uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_cp_128x256b_pair(uint32_t tmem_dst, uint64_t desc_src) {
  asm volatile("tcgen05.cp.cta_group::2.128x256b [%0], %1;" ::"r"(tmem_dst), "l"(desc_src) : "memory");
}

// K-major operand tile in shared memory, 128-byte swizzle: rows of 128 B, 8-row groups 1024 B apart.
// (cute::UMMA::SmemDescriptor: start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46), version=1 [46,48),
// layout SWIZZLE_128B=2 [61,64).)
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFF) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) |
         (2ull << 61);
}
// kind::f16 instruction descriptor (cute::UMMA::InstrDescriptor): D=f32 [4,6)=1, A=B=f16 (0),
// both K-major (0), N>>3 at [17,23), M>>4 at [24,29).
__host__ __device__ constexpr uint32_t instr_desc_f16(int m, int n) {
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// Keep the KSUB = 4 smallest offered (score, prototype index) pairs of one (row, epilogue warp) in shared
// memory: four scores (one 16-byte word; +inf = free slot) and their four prototype indices (INT_MAX for a
// free slot).  Pairs are ordered by score, then by prototype index, so among exact duplicates -- identical
// shadows give bit-identical scores -- the lowest index always survives, which is the tie rule of the
// reference (sklearn/utils/_heap.pyx:46).  Returns {gate score, gate index, out}: the gate is the largest
// pair in the table afterwards -- a later pair above it cannot enter, so the caller folds such a score (or
// the minimum of a whole chunk) into `evicted` without calling; out = the score that left or did not fit
// (+inf if none).  Not inlined (rare); everything it touches is shared memory or registers: the first
// version looked the prototype index up in global memory and kept its counters on the stack, ~1000 cycles
// of latency per call, which on maps with many near-identical prototypes (17 M calls per million rows late
// in a fit, most of them exact score ties) stalled the epilogue behind the two accumulator buffers and
// tripled K1.
__device__ __forceinline__ float4 lds_f4(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ int4 lds_i4(uint32_t a) {
  int4 v;
  asm volatile("ld.shared.v4.s32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts_f1(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void sts_i1(uint32_t a, int v) { asm volatile("st.shared.s32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ bool pair_after(float va, int ja, float vb, int jb) {  // (va, ja) > (vb, jb)
  return va > vb || (va == vb && ja > jb);
}

// Per-CTA constants of the epilogue, kept in shared memory so that slow_offer needs few arguments.
struct EpiConst {
  const int32_t* proto_of_col;
  uint32_t pstride, mpad;
  int any_order;
};
constexpr uint32_t kTabIdxOffset = 128 * 4 * 4 * 4;  // BM * EPI_SUBS * KSUB * 4: scores -> indices of the same table

// Offer (s, shadow column) to the table at val_addr.  Returns {fast gate, out}: `out` is the score that left
// the table or did not fit (+inf if none); the FAST GATE g lets the caller skip the call: a later score >= g
// cannot enter.  With any_order (equal scores need no index order, see dbgsom_exclude_duplicates) g is the
// largest score in the table, otherwise the next float above it, so that an exact tie still comes here and is
// decided by the prototype index.  +inf while a slot is free.
__device__ __noinline__ float2 slow_offer(float s, int col, uint32_t val_addr, uint32_t const_addr) {
  const EpiConst* ec;
  {
    uint64_t g;
    asm volatile("cvta.shared.u64 %0, %1;" : "=l"(g) : "l"((uint64_t)const_addr));
    ec = reinterpret_cast<const EpiConst*>(g);
  }
  const uint32_t idx_addr = val_addr + kTabIdxOffset;
  const int j = ec->pstride ? (int)(((uint32_t)col * ec->pstride) % ec->mpad) : ec->proto_of_col[col];
  const float4 v4 = lds_f4(val_addr);
  const int4 j4 = lds_i4(idx_addr);
  float v0 = v4.x, v1 = v4.y, v2 = v4.z, v3 = v4.w;
  int c0 = j4.x, c1 = j4.y, c2 = j4.z, c3 = j4.w;
  // largest pair of the table (scalars only: indexed local arrays would live in local memory)
  int w = 0;
  float wv = v0;
  int wc = c0;
  if (pair_after(v1, c1, wv, wc)) { w = 1; wv = v1; wc = c1; }
  if (pair_after(v2, c2, wv, wc)) { w = 2; wv = v2; wc = c2; }
  if (pair_after(v3, c3, wv, wc)) { w = 3; wv = v3; wc = c3; }
  const bool replace = pair_after(wv, wc, s, j);
  const float out = replace ? wv : s;  // +inf when a free slot was taken: a no-op for the caller's minimum
  if (replace) {
    sts_f1(val_addr + 4 * w, s);
    sts_i1(idx_addr + 4 * w, j);
    if (w == 0) v0 = s;
    if (w == 1) v1 = s;
    if (w == 2) v2 = s;
    if (w == 3) v3 = s;
  }
  float g = fmaxf(fmaxf(v0, v1), fmaxf(v2, v3));
  if (!ec->any_order && g < 3.0e38f) g = nextafterf(g, __int_as_float(0x7f800000));
  return make_float2(g, out);
}

// Top-k form of slow_offer: insert (s, shadow column) into the sorted table at val_addr (slot q at + q * BM * 4) whose
// first k slots are in use (+inf / INT_MAX = free).  Returns {gate, out}: gate = the k-th pair's score (+inf while a
// slot is free) -- a later score above it cannot enter; out = the score that left the table or did not enter.
__device__ __noinline__ float2 slow_offer_topk(float s, int col, uint32_t val_addr, uint32_t const_addr, int k) {
  const EpiConst* ec;
  {
    uint64_t g;
    asm volatile("cvta.shared.u64 %0, %1;" : "=l"(g) : "l"((uint64_t)const_addr));
    ec = reinterpret_cast<const EpiConst*>(g);
  }
  const uint32_t idx_addr = val_addr + kTopIdxOffset;
  const int j = ec->pstride ? (int)(((uint32_t)col * ec->pstride) % ec->mpad) : ec->proto_of_col[col];
  int pos = k - 1;
  float lv;
  int lj;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(lv) : "r"(val_addr + pos * BM * 4));
  asm volatile("ld.shared.s32 %0, [%1];" : "=r"(lj) : "r"(idx_addr + pos * BM * 4));
  if (!pair_after(lv, lj, s, j)) return make_float2(lv, s);  // (s, j) does not go before the k-th pair
  while (pos > 0) {
    float pv;
    int pj;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(pv) : "r"(val_addr + (pos - 1) * BM * 4));
    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(pj) : "r"(idx_addr + (pos - 1) * BM * 4));
    if (!pair_after(pv, pj, s, j)) break;
    sts_f1(val_addr + pos * BM * 4, pv);
    sts_i1(idx_addr + pos * BM * 4, pj);
    --pos;
  }
  sts_f1(val_addr + pos * BM * 4, s);
  sts_i1(idx_addr + pos * BM * 4, j);
  float g;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(g) : "r"(val_addr + (k - 1) * BM * 4) : "memory");
  return make_float2(g, lv);  // lv = +inf when a free slot was taken
}

// ------------------------------------------------------------------------------------------ layout
// RES_KB: k-blocks of the sample tile kept resident (0 = samples stream through the ring as well)
// ATM: the sample tile lives in TENSOR memory instead (columns [2*BN, 2*BN + 32*KB*NA)): its k-blocks pass
//      through the ring once per row tile and are moved with tcgen05.cp; the MMA then takes A from TMEM,
//      which leaves all shared memory to the prototype ring (5 stages instead of 2 at D = 256, 3 passes)
//      and, for D <= 128, tensor-memory room for three accumulator buffers instead of two.
// PAIRS: the streamed-operand form run as CTA pairs -- each CTA stages only its half of a prototype tile
template <int NPASS, int BN, int RES_KB, int AKB, bool PAIRS = false, int EXTRA_BYTES = 0>
struct Cfg {
  static constexpr bool ATM = AKB > 0;  // AKB: k-blocks of the sample tile held in tensor memory
  static constexpr bool XRES = RES_KB > 0;
  static constexpr bool ASTREAM = !XRES && !ATM;
  static constexpr int NA = NPASS == 3 ? 2 : 1;  // hi (+ lo) tiles per operand
  static constexpr int B_TILE_BYTES = BN * BK * 2;
  static_assert(!PAIRS || ASTREAM, "PAIRS is the streamed form");
  static constexpr int STAGE_BYTES = NA * (PAIRS ? B_TILE_BYTES / 2 : B_TILE_BYTES) + (ASTREAM ? NA * A_TILE_BYTES : 0);
  static_assert(!ATM || (RES_KB == 0 && B_TILE_BYTES <= A_TILE_BYTES), "TMEM-resident A shares the ring: BN <= 128");
  static constexpr int A_COLS = AKB * NA * (BK / 2);                 // tensor-memory columns of the sample tile
  // accumulator buffers; the streamed pair form with 128-column tiles closes its accumulation chain every few
  // k-blocks (SEGM in the kernel) and rotates through four partial accumulators
  static constexpr int NACC = ATM ? ((512 - A_COLS) / BN > 4 ? 4 : (512 - A_COLS) / BN) : (PAIRS && BN == 128 ? 4 : 2);
  static_assert(NACC >= 2, "need two accumulator buffers");
  static constexpr int RES_BYTES = RES_KB * NA * A_TILE_BYTES;
  // candidate tables [row][sub][KSUB] (idx + val), shared running minima [row], merge states [row][sub][4]
  static constexpr int RING_BYTES = BM * EPI_SUBS * KSUB * 8 + BM * 4 + BM * EPI_SUBS * 16;
  static constexpr int MISC_BYTES = 1024;  // barriers + tmem pointer
  static constexpr int WN_SMEM_FLOATS = ATM ? 4096 : 0;  // wnorm staged in shared memory when it fits
  static constexpr int WN_BYTES = WN_SMEM_FLOATS * 4;
  static constexpr int SMEM_BUDGET = 227 * 1024 - 1024;  // minus alignment slack
  // (with the sample tile in tensor memory the ring is cut into 16 KB slots, see the kernel: budget in those units)
  static constexpr int STAGE_UNIT = ATM ? (STAGE_BYTES > A_TILE_BYTES ? STAGE_BYTES : A_TILE_BYTES) : STAGE_BYTES;
  // EXTRA_BYTES: the FLAG pass of the selective search keeps one minimum per (32-column chunk, row) of a row tile
  static constexpr int STAGES_RAW = (SMEM_BUDGET - RES_BYTES - RING_BYTES - MISC_BYTES - WN_BYTES - EXTRA_BYTES) / STAGE_UNIT;
  static constexpr int STAGES = STAGES_RAW > (ATM ? 12 : 8) ? (ATM ? 12 : 8) : STAGES_RAW;
  static constexpr int RING_STAGE_BYTES = STAGES * STAGE_UNIT;  // bytes of the operand ring
  static constexpr int SMEM_BYTES = RES_BYTES + RING_STAGE_BYTES + RING_BYTES + MISC_BYTES + WN_BYTES + EXTRA_BYTES + 1024;
  static constexpr int TMEM_COLS = ATM ? 512 : NACC * BN;  // accumulator buffers (+ the sample tile)
  static_assert(STAGES >= 2, "not enough shared memory for a pipeline");
};

struct Barriers {
  uint64_t full[16], empty[16];
  uint64_t a_full, a_empty;
  uint64_t tmem_full[4], tmem_empty[4];
  uint32_t tmem_base;
  EpiConst epi;
};

// CL: thread-block cluster size (1, 2 or 4).  The CTAs of a cluster work on different row tiles in lock
// step and share every prototype tile: CTA r fetches rows [r * BN / CL, (r + 1) * BN / CL) of it and TMA
// multicasts them into all CL shared memories, so the L2 -> SM traffic of the prototype stream (the whole
// shadow matrix per 128 sample rows: 7 TB/s at config 3, which is what kept the tensor pipe at 78 %)
// drops by CL.  A ring stage is free again when the MMA warps of ALL CL CTAs have consumed it (their
// commits arrive on every CTA's `empty` barrier).
// SEL: 0 = the classic search over all column tiles; 1 = FLAG pass of the selective search (one fp16 pass, lean
// epilogue: per pair of row tiles, which column tiles hold a score inside the one-pass bound of one of its rows);
// 2 = REFINE pass (the classic three-pass search over exactly those column tiles).  Both need the CTA-pair form with
// the sample tile in tensor memory.  row_perm: the shadows are in sorted sample order (shadow row p = sample
// row_perm[p]); every per-sample read and write below goes through it.
// TB: per-tile error bounds (streamed forms, one winner).  tile_bound[2 q], [2 q + 1] = max ||u_j|| and max |wnorm_j|
// over shadow columns [128 q, 128 q + 128) (dbgsom_tile_bounds).  The rounding error of a score is proportional to the
// norm of ITS prototype, so a column of tile T is off by at most B_T = bound(||x'||, maxima of T) instead of the bound
// taken with the maxima of the whole map.  On large half-trained maps most prototypes form a flat sheet of small norm
// far from the samples while a few unfolded ones carry the maxima: thousands of sheet prototypes fell inside the
// global bound of a row and none of these rows could be proven a near-tie (2 B / d^2 ~ 1.1e-6 at the config-5 shape:
// 6 % of the rows went to the float64 re-scan of all prototypes, 3x the time of the search itself).  With tile bounds
// the tables work in KEY units, key = score - B_T (a lower bound of the exact score): a column is a candidate iff its
// key <= U, the smallest upper bound (score + B_T) seen so far, and a flagged row carries U2 - min key -- a proven
// bound on the exact best / second-best gap -- instead of the raw score gap.  Tile maxima are floored at 1/8 of the
// global ones: the coefficients were calibrated against global maxima (common.cuh), the floor keeps a margin.
constexpr float kTileBoundFloor = 0.125f;
// SGT > 0: segmented accumulation for the streamed pair form with 256-column MMAs, SGT k-blocks per chain.  An epilogue
// thread cannot hold the 64 running sums of a 256-column tile (96 registers at 640 threads), so the sums live in TENSOR
// memory: the two 256-column regions alternate as sum and partial accumulator -- the first chain of a tile accumulates
// into the sum region, every later chain into the other one, and the epilogue adds each partial into the sum with
// tcgen05.ld / tcgen05.st before handing the region back.  The regions swap roles per tile, so the final epilogue of
// a tile overlaps the first chain of the next.
template <int NPASS, int NB, int BN, int RES_KB, int AKB, int CL, bool PAIR = false, int SEL = 0, bool TB = false,
          int SGT = 0>
__global__ void __launch_bounds__(TC_THREADS, 1)
    bmu_cand_tensor_kernel(const __grid_constant__ CUtensorMap map_xh, const __grid_constant__ CUtensorMap map_xl,
                           const __grid_constant__ CUtensorMap map_wh, const __grid_constant__ CUtensorMap map_wl,
                           const __grid_constant__ CUtensorMap map_wb, const float* __restrict__ bias_scale,
                           int64_t N, int KB, int NT, const float* __restrict__ wnorm,
                           const int32_t* __restrict__ proto_of_col, int pstride, int ties_any,
                           const float* __restrict__ xnorm16,
                           const float* __restrict__ wmax, float bound_coef, float acc_coef,
                           int32_t* __restrict__ idx_out, int32_t* __restrict__ cand_idx,
                           uint8_t* __restrict__ cand_count, const int32_t* __restrict__ row_perm,
                           unsigned long long* __restrict__ tile_mask,
                           int fg_shift, unsigned long long* __restrict__ sel_stats,
                           const float* __restrict__ tile_bound, int n_topk) {
  static_assert(!TB || (NB == 1 && SEL == 0 && BN % 128 == 0), "tile bounds: classic one-winner search, 128-column granules");
  using C = Cfg<NPASS, BN, RES_KB, AKB, PAIR && AKB == 0 && RES_KB == 0, extra_bytes<NB, SEL>()>;
  static_assert(NB <= 2 || (NB == KTOP && SEL == 0 && NPASS == 3), "top-k: the classic three-pass search");
  static_assert(SEL == 0 || (PAIR && AKB > 0 && NB == 1 && NPASS == (SEL == 1 ? 1 : 3)),
                "selective search: CTA pairs, sample tile in tensor memory, one winner");
  constexpr bool ATM = C::ATM;
  static_assert(!PAIR || (CL == 2 && (ATM || C::ASTREAM)), "the CTA-pair form needs a cluster of two; sample tile in tensor memory or streamed");
  constexpr int B_PART_BYTES = PAIR ? C::B_TILE_BYTES / 2 : C::B_TILE_BYTES;  // prototype tile bytes per CTA and shadow
  // pair: the ring is cut into 16 KB slots -- one k-block of one sample shadow, or one k-block of my half of both
  // prototype shadows -- so the same shared memory holds twice as many k-blocks in flight
  // SEGM: segmented accumulation (streamed pair form, 128-column tiles).  The fp32 accumulator in tensor memory takes
  // one rounding per MMA, 768 of them per score at D = 4096, and the error bound had to grow with that chain
  // (common.cuh, tensor_acc_coef).  Here the MMA stream starts a fresh accumulator every SEG k-blocks (48 steps, the
  // chain of D = 256) and the epilogue sums the partial tiles in registers, so the bound of D = 256 (x2 for the
  // fp32 sums) holds for any D.
  constexpr bool SEGM = PAIR && C::ASTREAM && BN == 128;
  constexpr int SEG = 4;
  constexpr bool SEGT = SGT > 0;
  static_assert(!SEGT || (PAIR && C::ASTREAM && BN == 256 && C::NACC == 2 && SEL == 0), "tensor-memory sums: streamed pair form, 256 columns");
  static_assert(!SEGM || BN / 32 == EPI_SUBS, "segmented accumulation: one chunk per epilogue warp and tile");
  constexpr bool PAIR_ATM = PAIR && ATM;  // (the streamed pair form keeps whole stages: prototypes half + samples)
  constexpr int SLOT_BYTES = PAIR_ATM ? A_TILE_BYTES : C::STAGE_BYTES;
  constexpr int NSLOT = PAIR_ATM ? (C::RING_STAGE_BYTES / A_TILE_BYTES > 16 ? 16 : C::RING_STAGE_BYTES / A_TILE_BYTES)
                                 : C::STAGES;
  static_assert(!PAIR_ATM || C::NA * B_PART_BYTES <= SLOT_BYTES, "a prototype k-block of the pair form must fit a slot");
  constexpr int NACC = C::NACC;
  constexpr bool XRES = C::XRES;
  constexpr bool ASTREAM = C::ASTREAM;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* res_a = smem;                               // [kb][hi|lo] A tiles (XRES)
  uint8_t* stages = smem + C::RES_BYTES;               // ring
  // wnorm staging, or -- in bias mode -- the constant A tile of the bias k-step (1024-byte aligned for its descriptor)
  float* wn_smem = reinterpret_cast<float*>(stages + C::RING_STAGE_BYTES);
  uint8_t* ring = stages + C::RING_STAGE_BYTES + C::WN_BYTES;  // candidate tables
  Barriers* bars = reinterpret_cast<Barriers*>(ring + C::RING_BYTES);
  float* chunk_min = reinterpret_cast<float*>(ring + C::RING_BYTES + C::MISC_BYTES);  // [chunk][row] (FLAG pass only)
  float* top_val = chunk_min;  // top-k tables [sub][slot][row] (NB > 2 only; same region)
  float* tab_val = reinterpret_cast<float*>(ring);
  int* tab_idx = reinterpret_cast<int*>(ring + BM * EPI_SUBS * KSUB * 4);  // = tab_val + kTabIdxOffset bytes
  float* row_min = reinterpret_cast<float*>(ring + BM * EPI_SUBS * KSUB * 8);
  float4* sub_state = reinterpret_cast<float4*>(ring + BM * EPI_SUBS * KSUB * 8 + BM * 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int64_t n_row_tiles = ceil_div<int64_t>(N, BM);
  // row tile of iteration `it`: clusters stride over groups of CL consecutive tiles; every CTA of a cluster runs
  // the same number of iterations (tiles past the end are dummies: zero-filled loads, no output)
  const uint32_t cl_rank = CL > 1 ? cluster_ctarank() : 0u;
  const int64_t n_clusters = gridDim.x / CL;
  const int64_t cluster_id = blockIdx.x / CL;
  const int64_t n_iters = ceil_div<int64_t>(n_row_tiles, n_clusters * CL);
  constexpr uint16_t cl_mask = (uint16_t)((1u << CL) - 1u);
  auto tile_of = [&](int64_t it) { return (it * n_clusters + cluster_id) * CL + cl_rank; };
  // selective search: masks and start tiles are kept per PAIR of row tiles (one cluster iteration)
  const int64_t n_pairs = ceil_div<int64_t>(n_row_tiles, 2);
  auto pair_of = [&](int64_t it) { return it * n_clusters + cluster_id; };
  // column tiles of row-tile iteration `it`: all NT in order (classic, FLAG) or the set bits of the pair's mask (REFINE).  Every warp role derives the same sequence from global memory.
  auto sel_mask = [&](int64_t it) -> unsigned long long {
    const int64_t pr = pair_of(it);
    return (SEL == 2 && pr < n_pairs) ? tile_mask[pr] : 0ull;
  };

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_xh);
    tma_prefetch_desc(&map_wh);
    if (NPASS == 3) {
      tma_prefetch_desc(&map_xl);
      tma_prefetch_desc(&map_wl);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < NSLOT; ++s) {
      mbar_init(&bars->full[s], PAIR ? 2 : 1);   // pair: the leader's expect_tx arrive + the peer producer's arrive
      mbar_init(&bars->empty[s], PAIR ? 1 : CL);  // pair: one MMA stream frees the stage in both CTAs
    }
    mbar_init(&bars->a_full, 1);
    mbar_init(&bars->a_empty, 1);
    for (int b = 0; b < NACC; ++b) {
      mbar_init(&bars->tmem_full[b], 1);
      mbar_init(&bars->tmem_empty[b], PAIR ? 2 * EPI_WARPS : EPI_THREADS);  // pair: one arrive per epilogue warp of both CTAs
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars->tmem_base)),
                   "r"((uint32_t)C::TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars->tmem_base)),
                   "r"((uint32_t)C::TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  // bias mode (CTA pairs only): wnorm enters the accumulator through one extra k-step per output tile
  // (dbgsom_prepare_bias).  Its A operand is constant: E = bias_scale[0] in the first three columns of every row, a
  // 128 x 64 fp16 K-major tile with the 128-byte swizzle (16-byte chunk c of row r sits at chunk c ^ (r & 7)).
  const float bias_E = (PAIR && bias_scale != nullptr) ? bias_scale[0] : 0.f;
  const bool bias_mode = PAIR && bias_E > 0.f;
  if (bias_mode) {
    const uint32_t e16 = (uint32_t)__half_as_ushort(__float2half_rn(bias_E));
    uint4* tile = reinterpret_cast<uint4*>(wn_smem);
    for (int q = threadIdx.x; q < BM * 8; q += TC_THREADS) {
      const int r = q >> 3, ch = q & 7;
      tile[q] = ch == (r & 7) ? make_uint4(e16 | (e16 << 16), e16, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> tensor-core reads
  }
  tc_fence_before();
  __syncthreads();
  if (CL > 1) cluster_sync_all();  // every CTA's barriers exist before a peer signals them
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  if (warp == 0) {
    // ================================================================ TMA producer
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0, a_phase = 0;
      unsigned long long sel_tiles = 0, sel_pairs = 0;
      unsigned long long pmask_next = SEL == 2 ? sel_mask(0) : 0ull;
      for (int64_t it = 0; it < n_iters; ++it) {
        const int row0 = (int)(tile_of(it) * BM);
        const unsigned long long pmask_it = pmask_next;
        if (SEL == 2) pmask_next = it + 1 < n_iters ? sel_mask(it + 1) : 0ull;
        if (XRES) {
          mbar_wait(&bars->a_empty, a_phase ^ 1);
          mbar_expect_tx(&bars->a_full, (uint32_t)(KB * C::NA * A_TILE_BYTES));
          for (int kb = 0; kb < KB; ++kb) {
            tma_load_2d(res_a + (kb * C::NA + 0) * A_TILE_BYTES, &map_xh, &bars->a_full, kb * BK, row0);
            if (NPASS == 3) tma_load_2d(res_a + (kb * C::NA + 1) * A_TILE_BYTES, &map_xl, &bars->a_full, kb * BK, row0);
          }
          a_phase ^= 1;
        }
        if (ATM) {  // the sample tile's k-blocks travel through the ring once per row tile
          for (int kb = 0; kb < KB; ++kb) {
            if (PAIR) {  // one slot per shadow; both CTAs' bytes are counted on the leader's barrier
              for (int h = 0; h < C::NA; ++h) {
                mbar_wait(&bars->empty[stage], phase ^ 1);
                const uint32_t lead_full = mapa_u32(smem_u32(&bars->full[stage]), 0);
                if (cl_rank == 0) mbar_expect_tx(&bars->full[stage], (uint32_t)(2 * A_TILE_BYTES));
                else mbar_arrive_cluster(lead_full);
                tma_load_2d_pair(stages + stage * SLOT_BYTES, h == 0 ? &map_xh : &map_xl, lead_full, kb * BK, row0);
                if (++stage == NSLOT) {
                  stage = 0;
                  phase ^= 1;
                }
              }
              continue;
            }
            mbar_wait(&bars->empty[stage], phase ^ 1);
            uint8_t* st = stages + stage * C::STAGE_BYTES;
            mbar_expect_tx(&bars->full[stage], (uint32_t)(C::NA * A_TILE_BYTES));
            tma_load_2d(st, &map_xh, &bars->full[stage], kb * BK, row0);
            if (NPASS == 3) tma_load_2d(st + A_TILE_BYTES, &map_xl, &bars->full[stage], kb * BK, row0);
            if (++stage == C::STAGES) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
        unsigned long long selm = pmask_it;
        const int n_sel = SEL == 2 ? __popcll(selm) : NT;
        if (SEL == 2 && cl_rank == 0 && pair_of(it) < n_pairs) {
          sel_tiles += (unsigned)n_sel;
          ++sel_pairs;
        }
        for (int ti = 0; ti < n_sel; ++ti) {
          int nt = ti;
          if (SEL == 2) {
            nt = __ffsll((long long)selm) - 1;
            selm &= selm - 1;
          }
          for (int kb = 0; kb < KB; ++kb) {
            mbar_wait(&bars->empty[stage], phase ^ 1);
            uint8_t* st = stages + stage * SLOT_BYTES;
            if (PAIR) {  // my half of the prototype tile (rows [rank * BN/2, +BN/2)) into MY shared memory only
              const uint32_t lead_full = mapa_u32(smem_u32(&bars->full[stage]), 0);
              if (cl_rank == 0) mbar_expect_tx(&bars->full[stage], (uint32_t)(2 * (C::NA * B_PART_BYTES + (ASTREAM ? C::NA * A_TILE_BYTES : 0))));
              else mbar_arrive_cluster(lead_full);
              const int prow = nt * BN + (int)cl_rank * (BN / 2);
              tma_load_2d_pair(st, &map_wh, lead_full, kb * BK, prow);
              if (NPASS == 3) tma_load_2d_pair(st + B_PART_BYTES, &map_wl, lead_full, kb * BK, prow);
              if (ASTREAM) {  // my own sample rows, this k-block
                uint8_t* sa = st + C::NA * B_PART_BYTES;
                tma_load_2d_pair(sa, &map_xh, lead_full, kb * BK, row0);
                if (NPASS == 3) tma_load_2d_pair(sa + A_TILE_BYTES, &map_xl, lead_full, kb * BK, row0);
              }
              if (++stage == NSLOT) {
                stage = 0;
                phase ^= 1;
              }
              continue;
            }
            mbar_expect_tx(&bars->full[stage], (uint32_t)C::STAGE_BYTES);
            if (CL == 1) {
              tma_load_2d(st, &map_wh, &bars->full[stage], kb * BK, nt * BN);
              if (NPASS == 3) tma_load_2d(st + C::B_TILE_BYTES, &map_wl, &bars->full[stage], kb * BK, nt * BN);
            } else {  // my 1/CL of the prototype tile, to everybody
              const int part = C::B_TILE_BYTES / CL, prow = nt * BN + (int)cl_rank * (BN / CL);
              tma_load_2d_mc(st + cl_rank * part, &map_wh, &bars->full[stage], kb * BK, prow, cl_mask);
              if (NPASS == 3)
                tma_load_2d_mc(st + C::B_TILE_BYTES + cl_rank * part, &map_wl, &bars->full[stage], kb * BK, prow, cl_mask);
            }
            if (ASTREAM) {
              uint8_t* sa = st + C::NA * C::B_TILE_BYTES;
              tma_load_2d(sa, &map_xh, &bars->full[stage], kb * BK, row0);
              if (NPASS == 3) tma_load_2d(sa + A_TILE_BYTES, &map_xl, &bars->full[stage], kb * BK, row0);
            }
            if (++stage == C::STAGES) {
              stage = 0;
              phase ^= 1;
            }
          }
          if (PAIR && bias_mode) {  // my half of the tile's bias rows: one more slot
            mbar_wait(&bars->empty[stage], phase ^ 1);
            const uint32_t lead_full = mapa_u32(smem_u32(&bars->full[stage]), 0);
            if (cl_rank == 0) mbar_expect_tx(&bars->full[stage], (uint32_t)(2 * B_PART_BYTES));
            else mbar_arrive_cluster(lead_full);
            tma_load_2d_pair(stages + stage * SLOT_BYTES, &map_wb, lead_full, 0, nt * BN + (int)cl_rank * (BN / 2));
            if (++stage == NSLOT) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
      }
      if (SEL == 2 && sel_stats != nullptr && sel_pairs) {
        atomicAdd(sel_stats + 0, sel_tiles);
        atomicAdd(sel_stats + 1, sel_pairs);
      }
    }
  } else if (warp == 1 && (!PAIR || cl_rank == 0)) {
    // ================================================================ MMA issuer (pair: the leader CTA only)
    if (elect_one()) {
      constexpr uint32_t idesc = instr_desc_f16(PAIR ? 2 * BM : BM, BN);
      int stage = 0;
      uint32_t phase = 0, a_phase = 0, acc = 0, acc_phase = 0;
      uint32_t rph = 0;  // SEGT: phase bit of each tensor-memory region (acc = the sum region of the current tile)
      unsigned long long mask_next = SEL == 2 ? sel_mask(0) : 0ull;  // the pair's mask is loaded one row tile ahead
      for (int64_t it = 0; it < n_iters; ++it) {
        const unsigned long long mask_it = mask_next;
        if (SEL == 2) mask_next = it + 1 < n_iters ? sel_mask(it + 1) : 0ull;
        if (XRES) {
          mbar_wait(&bars->a_full, a_phase);
          a_phase ^= 1;
        }
        const uint32_t tmem_a = tmem_base + NACC * BN;  // ATM: [kb][k] -> 8 columns each, lo half after AKB blocks
        if (ATM) {
          // tcgen05.cp and tcgen05.mma execute in issue order, so these copies run after the previous row
          // tile's MMAs have read the old sample tile and before this row tile's MMAs read the new one
          for (int kb = 0; kb < KB; ++kb) {
            if (PAIR) {  // one slot per shadow; each CTA's staged rows go to its own tensor memory
              for (int h = 0; h < C::NA; ++h) {
                mbar_wait(&bars->full[stage], phase);
                tc_fence_after();
                const uint32_t sa = smem_u32(stages + stage * SLOT_BYTES);
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k)
                  tc_cp_128x256b_pair(tmem_a + h * AKB * (BK / 2) + kb * (BK / 2) + k * 8,
                                      smem_desc_sw128(sa + k * UMMA_K * 2));
                tc_commit_pair(&bars->empty[stage], cl_mask);
                if (++stage == NSLOT) {
                  stage = 0;
                  phase ^= 1;
                }
              }
              continue;
            }
            mbar_wait(&bars->full[stage], phase);
            tc_fence_after();
            const uint32_t sa = smem_u32(stages + stage * C::STAGE_BYTES);
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              tc_cp_128x256b(tmem_a + kb * (BK / 2) + k * 8, smem_desc_sw128(sa + k * UMMA_K * 2));
              if (NPASS == 3)
                tc_cp_128x256b(tmem_a + AKB * (BK / 2) + kb * (BK / 2) + k * 8,
                               smem_desc_sw128(sa + A_TILE_BYTES + k * UMMA_K * 2));
            }
            if (CL == 1) tc_commit(&bars->empty[stage]); else tc_commit_mc(&bars->empty[stage], cl_mask);
            if (++stage == C::STAGES) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
        const int n_sel = SEL == 2 ? __popcll(mask_it) : NT;
        for (int nt = 0; nt < n_sel; ++nt) {
          uint32_t tmem_d = tmem_base + acc * BN;
          if (!SEGM && !SEGT) {
            mbar_wait(&bars->tmem_empty[acc], acc_phase ^ 1);
            tc_fence_after();
          }
          uint32_t region = acc;
          for (int kb = 0; kb < KB; ++kb) {
            if (SEGM && kb % SEG == 0) {  // a fresh partial accumulator
              mbar_wait(&bars->tmem_empty[acc], acc_phase ^ 1);
              tc_fence_after();
              tmem_d = tmem_base + acc * BN;
            }
            if (SEGT && kb % (SEGT ? SGT : 1) == 0) {  // a fresh chain: into the sum region first, then into the other one
              region = kb == 0 ? acc : acc ^ 1u;
              mbar_wait(&bars->tmem_empty[region], ((rph >> region) & 1u) ^ 1u);
              tc_fence_after();
              tmem_d = tmem_base + region * BN;
            }
            mbar_wait(&bars->full[stage], phase);
            tc_fence_after();
            uint8_t* st = stages + stage * SLOT_BYTES;
            const uint32_t b_hi = smem_u32(st);
            const uint32_t b_lo = b_hi + B_PART_BYTES;
            const uint32_t a_hi = XRES ? smem_u32(res_a + kb * C::NA * A_TILE_BYTES)
                                       : smem_u32(st + C::NA * B_PART_BYTES);
            const uint32_t a_lo = a_hi + A_TILE_BYTES;
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              const uint32_t koff = k * UMMA_K * 2;  // bytes along K inside the swizzle atom
              if (PAIR && ASTREAM) {  // both operands from shared memory, each CTA's own sample rows
                tc_mma_f16_ss_pair(tmem_d, smem_desc_sw128(a_hi + koff), smem_desc_sw128(b_hi + koff), idesc,
                                   ((SEGM ? kb % SEG : SEGT ? kb % (SEGT ? SGT : 1) : kb) | k) != 0);
                if (NPASS == 3) {
                  tc_mma_f16_ss_pair(tmem_d, smem_desc_sw128(a_hi + koff), smem_desc_sw128(b_lo + koff), idesc, 1);
                  tc_mma_f16_ss_pair(tmem_d, smem_desc_sw128(a_lo + koff), smem_desc_sw128(b_hi + koff), idesc, 1);
                }
              } else if (PAIR) {
                const uint32_t ta_hi = tmem_a + kb * (BK / 2) + k * 8;
                const uint32_t ta_lo = ta_hi + AKB * (BK / 2);
                tc_mma_f16_ts_pair(tmem_d, ta_hi, smem_desc_sw128(b_hi + koff), idesc, (kb | k) != 0);
                if (NPASS == 3) {
                  tc_mma_f16_ts_pair(tmem_d, ta_hi, smem_desc_sw128(b_lo + koff), idesc, 1);
                  tc_mma_f16_ts_pair(tmem_d, ta_lo, smem_desc_sw128(b_hi + koff), idesc, 1);
                }
              } else if (ATM) {
                const uint32_t ta_hi = tmem_a + kb * (BK / 2) + k * 8;
                const uint32_t ta_lo = ta_hi + AKB * (BK / 2);
                tc_mma_f16_ts(tmem_d, ta_hi, smem_desc_sw128(b_hi + koff), idesc, (kb | k) != 0);
                if (NPASS == 3) {
                  tc_mma_f16_ts(tmem_d, ta_hi, smem_desc_sw128(b_lo + koff), idesc, 1);
                  tc_mma_f16_ts(tmem_d, ta_lo, smem_desc_sw128(b_hi + koff), idesc, 1);
                }
              } else {
                tc_mma_f16(tmem_d, smem_desc_sw128(a_hi + koff), smem_desc_sw128(b_hi + koff), idesc, (kb | k) != 0);
                if (NPASS == 3) {
                  tc_mma_f16(tmem_d, smem_desc_sw128(a_hi + koff), smem_desc_sw128(b_lo + koff), idesc, 1);
                  tc_mma_f16(tmem_d, smem_desc_sw128(a_lo + koff), smem_desc_sw128(b_hi + koff), idesc, 1);
                }
              }
            }
            // frees the smem stage (in every CTA of the cluster) once these MMAs have read it
            if (PAIR) tc_commit_pair(&bars->empty[stage], cl_mask);
            else if (CL == 1) tc_commit(&bars->empty[stage]); else tc_commit_mc(&bars->empty[stage], cl_mask);
            if (++stage == NSLOT) {
              stage = 0;
              phase ^= 1;
            }
            if (SEGT && (kb % (SEGT ? SGT : 1) == (SEGT ? SGT : 1) - 1 || kb == KB - 1)) {  // chain complete
              tc_commit_pair(&bars->tmem_full[region], cl_mask);
              rph ^= 1u << region;
            }
            if (SEGM && kb % SEG == SEG - 1 && kb != KB - 1) {  // partial accumulator complete (the last one below)
              tc_commit_pair(&bars->tmem_full[acc], cl_mask);
              if (++acc == NACC) {
                acc = 0;
                acc_phase ^= 1;
              }
            }
          }
          if (PAIR && bias_mode) {  // + E * (h + m + l) = -wnorm / 2: the accumulator is now -score / 2
            mbar_wait(&bars->full[stage], phase);
            tc_fence_after();
            tc_mma_f16_ss_pair(tmem_d, smem_desc_sw128(smem_u32(wn_smem)), smem_desc_sw128(smem_u32(stages + stage * SLOT_BYTES)),
                               idesc, 1);
            tc_commit_pair(&bars->empty[stage], cl_mask);
            if (++stage == NSLOT) {
              stage = 0;
              phase ^= 1;
            }
          }
          // accumulator complete -> epilogue (pair: of both CTAs)
          if (SEGT) {
          } else if (PAIR) tc_commit_pair(&bars->tmem_full[acc], cl_mask); else tc_commit(&bars->tmem_full[acc]);
          if (++acc == NACC) {
            acc = 0;
            acc_phase ^= 1;
          }
        }
        if (XRES) tc_commit(&bars->a_empty);  // resident A tile may be overwritten
      }
    }
  } else if (warp >= EPI_WARP0) {
    // ================================================================ epilogue
    const int quarter = warp & 3;                  // TMEM lanes [32 * quarter, +32)
    const int sub = (warp - EPI_WARP0) >> 2;       // which of the four warps of this quarter
    const int t = quarter * 32 + lane;             // TMEM lane = row within the tile
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    static_assert(KSUB == 4 && BM * EPI_SUBS * KSUB * 4 == kTabIdxOffset, "slow_offer handles four-entry tables");
    const uint32_t my_val_addr = smem_u32(tab_val + (t * EPI_SUBS + sub) * KSUB);  // scores of my entries
    const uint32_t my_idx_addr = my_val_addr + kTabIdxOffset;                      // their prototype indices
    // equal scores need no index order when exact copies have left the search (dbgsom_exclude_duplicates)
    const bool any_order = NB == 1 && ties_any != 0;
    if (threadIdx.x == EPI_WARP0 * 32) {
      bars->epi.proto_of_col = proto_of_col;
      bars->epi.pstride = (uint32_t)pstride;
      bars->epi.mpad = (uint32_t)(NT * BN);
      bars->epi.any_order = any_order ? 1 : 0;
    }
    const uint32_t epi_const_addr = smem_u32(&bars->epi);
    // top-k: my table, slot q at + q * BM * 4 (values; indices kTopIdxOffset further)
    const uint32_t my_top_addr = smem_u32(top_val + sub * KTOP * BM + t);
    constexpr int CHUNKS = BN / 32;
    constexpr float kInf = 3.0e38f;
    if (sub == 0) row_min[t] = kInf;
    // wnorm is read by every row for every chunk: keep it in shared memory when it fits (global / L1
    // loads showed up as the longest stall of the epilogue at D = 128)
    const int mpad = NT * BN;
    const bool wn_in_smem = !bias_mode && C::WN_SMEM_FLOATS > 0 && mpad <= C::WN_SMEM_FLOATS;
    if (wn_in_smem)
      for (int i = threadIdx.x - EPI_WARP0 * 32; i < mpad; i += EPI_THREADS) wn_smem[i] = wnorm[i];
    const float* wn_src = wn_in_smem ? wn_smem : wnorm;
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS));
    uint32_t acc = 0, acc_phase = 0;
    uint32_t eph = 0;  // SEGT: phase bit of each tensor-memory region, epilogue side
    (void)eph;
    if constexpr (SEL == 1) {
      // ------------------------------------------------------------ FLAG pass: lean epilogue, no candidate tables
      // Per 32-column chunk a thread (= sample row) forms its 32 one-pass scores and stores their minimum in shared
      // memory, [chunk][row].  After the last column tile the row's smallest one-pass score is known, and with it the
      // FINAL bound: every chunk whose minimum lies inside it sets the bit of its column tile.  (Testing against the
      // running minimum instead flagged ~2x as many tiles: the bound is ~1e-3 of the score spread, so a running
      // minimum that is not yet the final one lets whole neighbourhoods through.)  The bits of a row-tile pair are
      // OR-ed over rows, warps and both CTAs into tile_mask.
      uint32_t* cta_mask = reinterpret_cast<uint32_t*>(sub_state);  // two words, zero between row tiles
      float* sub_min = reinterpret_cast<float*>(sub_state) + 4;      // [row][sub] minima of the four warps of a row
      if (threadIdx.x == EPI_WARP0 * 32) cta_mask[0] = cta_mask[1] = 0u;
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS));
      const int n_chunks = NT * CHUNKS;
      for (int64_t it = 0; it < n_iters; ++it) {
        const int64_t row = tile_of(it) * BM + t;
        const bool valid = row < N;
        const int64_t orow = valid ? (row_perm ? (int64_t)row_perm[row] : row) : 0;
        const float tau = valid ? 2.f * tensor_score_bound(xnorm16[orow], wmax, bound_coef, acc_coef) : 0.f;
        float m1 = kInf;
        for (int nt = 0; nt < NT; ++nt) {
          mbar_wait(&bars->tmem_full[acc], acc_phase);
          tc_fence_after();
          const uint32_t tmem_acc = tmem_base + lane_base + acc * BN;
#pragma unroll 1
          for (int c = (sub - nt * CHUNKS) & (EPI_SUBS - 1); c < CHUNKS; c += EPI_SUBS) {
            uint32_t r[32];
            tmem_ld_32x32(tmem_acc + c * 32, r);
            float a1;
            if (bias_mode) {
              // wnorm came in through the bias k-step: the accumulator is -score / 2, so the chunk's smallest score is
              // -2 x its largest accumulator -- no per-column load, no FFMA (at D = 128 this epilogue, not the MMA
              // stream, set the pace of the FLAG pass)
              tmem_ld_wait();
              float gmx[8];
#pragma unroll
              for (int g = 0; g < 8; ++g)
                gmx[g] = fmaxf(fmaxf(__uint_as_float(r[4 * g + 0]), __uint_as_float(r[4 * g + 1])),
                               fmaxf(__uint_as_float(r[4 * g + 2]), __uint_as_float(r[4 * g + 3])));
              a1 = -2.f * fmaxf(fmaxf(fmaxf(gmx[0], gmx[1]), fmaxf(gmx[2], gmx[3])),
                                fmaxf(fmaxf(gmx[4], gmx[5]), fmaxf(gmx[6], gmx[7])));
            } else {
              const int col = nt * BN + c * 32;
              const float4* wn4 = reinterpret_cast<const float4*>(wn_src + col);
              float4 w4[8];
#pragma unroll
              for (int g = 0; g < 8; ++g) w4[g] = wn4[g];
              tmem_ld_wait();
              float gmn[8];
#pragma unroll
              for (int g = 0; g < 8; ++g) {
                const float s0 = fmaf(-2.f, __uint_as_float(r[4 * g + 0]), w4[g].x);
                const float s1 = fmaf(-2.f, __uint_as_float(r[4 * g + 1]), w4[g].y);
                const float s2 = fmaf(-2.f, __uint_as_float(r[4 * g + 2]), w4[g].z);
                const float s3 = fmaf(-2.f, __uint_as_float(r[4 * g + 3]), w4[g].w);
                gmn[g] = fminf(fminf(s0, s1), fminf(s2, s3));
              }
              a1 = fminf(fminf(fminf(gmn[0], gmn[1]), fminf(gmn[2], gmn[3])),
                         fminf(fminf(gmn[4], gmn[5]), fminf(gmn[6], gmn[7])));
            }
            chunk_min[(nt * CHUNKS + c) * BM + t] = a1;
            m1 = fminf(m1, a1);
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&bars->tmem_empty[acc]), 0));
          if (++acc == NACC) {
            acc = 0;
            acc_phase ^= 1;
          }
        }
        sub_min[t * EPI_SUBS + sub] = m1;
        asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS));
        const float4 sm4 = *reinterpret_cast<const float4*>(sub_min + t * EPI_SUBS);
        const float thr = fminf(fminf(sm4.x, sm4.y), fminf(sm4.z, sm4.w)) + tau;
        uint32_t mlo = 0u, mhi = 0u;
        if (valid) {
          for (int ch = sub; ch < n_chunks; ch += EPI_SUBS) {
            const uint32_t bit = (uint32_t)(ch * 32) >> fg_shift;
            const uint32_t inb = chunk_min[ch * BM + t] <= thr ? 1u : 0u;
            mlo |= bit < 32u ? inb << bit : 0u;
            mhi |= bit >= 32u ? inb << (bit - 32u) : 0u;
          }
        }
        mlo = __reduce_or_sync(kFullMask, mlo);
        mhi = __reduce_or_sync(kFullMask, mhi);
        if (lane == 0) {
          if (mlo) atomicOr(&cta_mask[0], mlo);
          if (mhi) atomicOr(&cta_mask[1], mhi);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS));
        if (threadIdx.x == EPI_WARP0 * 32) {
          const unsigned long long m64 = (unsigned long long)cta_mask[0] | ((unsigned long long)cta_mask[1] << 32);
          const int64_t pr = pair_of(it);
          if (m64 && pr < n_pairs) atomicOr(tile_mask + pr, m64);
          cta_mask[0] = cta_mask[1] = 0u;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS));
      }
    } else {
    // Per row tile an epilogue thread needs its sample's index (through the permutation), the sample's norm (through that
    // index) and the pair's column-tile mask: three global loads, two of them dependent, which stalled every epilogue
    // warp at the start of every row tile (9 % of the REFINE pass's stall samples; it visits only ~10 column tiles per row
    // tile).  They are software-pipelined: the index two row tiles ahead, norm and mask one row tile ahead -- no load
    // is consumed in the iteration that issues it.
    auto fetch_orow = [&](int64_t it_) -> int64_t {
      const int64_t r_ = it_ < n_iters ? tile_of(it_) * BM + t : N;
      return r_ < N ? (row_perm ? (int64_t)row_perm[r_] : r_) : -1;
    };
    auto fetch_mask = [&](int64_t it_) -> unsigned long long { return it_ < n_iters ? sel_mask(it_) : 0ull; };
    int64_t orow_n1 = fetch_orow(0);               // index of my row in row tile it + 1 (it = -1 here)
    int64_t orow_n2 = fetch_orow(1);               //                                it + 2
    float xn_n1 = orow_n1 >= 0 ? xnorm16[orow_n1] : 0.f;
    unsigned long long mask_n1 = fetch_mask(0);
    for (int64_t it = 0; it < n_iters; ++it) {
      const int64_t row = tile_of(it) * BM + t;
      const int64_t orow = orow_n1 >= 0 ? orow_n1 : 0;
      const float tau = row < N ? 2.f * tensor_score_bound(xn_n1, wmax, bound_coef, acc_coef) : 0.f;
      const float xn_row = row < N ? xn_n1 : 0.f;
      unsigned long long selm = mask_n1;
      orow_n1 = orow_n2;
      xn_n1 = orow_n1 >= 0 ? xnorm16[orow_n1] : 0.f;  // address known since the previous iteration
      orow_n2 = fetch_orow(it + 2);
      mask_n1 = fetch_mask(it + 1);
      float m1 = kInf, m2 = kInf, thr = kInf, evicted = __int_as_float(0x7f800000);
      float gate = __int_as_float(0x7f800000);  // fast gate of my table (see slow_offer); +inf while a slot is free
      asm volatile("st.shared.v4.f32 [%0], {%1,%1,%1,%1};" ::"r"(my_val_addr), "f"(gate) : "memory");
      asm volatile("st.shared.v4.s32 [%0], {%1,%1,%1,%1};" ::"r"(my_idx_addr), "r"(0x7fffffff) : "memory");
      if constexpr (NB > 2) {
        for (int q = 0; q < n_topk; ++q) {
          sts_f1(my_top_addr + q * BM * 4, gate);
          sts_i1(my_top_addr + kTopIdxOffset + q * BM * 4, 0x7fffffff);
        }
      }
      const int n_sel = SEL == 2 ? __popcll(selm) : NT;
      for (int ti = 0; ti < n_sel; ++ti) {
        int nt = ti;
        if (SEL == 2) {
          nt = __ffsll((long long)selm) - 1;
          selm &= selm - 1;
        }
        float kb = 0.f;  // TB: the bound of this column tile for my row (keys = score - kb); 0 otherwise
        if (TB) {
          const float* tb = tile_bound + 2 * (nt * (BN / 128));
          float um = tb[0], wm = tb[1];
#pragma unroll
          for (int q = 1; q < BN / 128; ++q) {
            um = fmaxf(um, tb[2 * q]);
            wm = fmaxf(wm, tb[2 * q + 1]);
          }
          um = fmaxf(um, kTileBoundFloor * wmax[0]);
          wm = fmaxf(wm, kTileBoundFloor * wmax[2]);
          const float xw = xn_row * um;
          kb = xw * bound_coef + acc_coef * (xw + wm);
        }
        if constexpr (SEGT) {
          // sums in tensor memory: region `acc` holds the first chain of this tile, every later chain arrives in the
          // other region and is added in (my chunks only), 16 columns at a time
          const uint32_t R = acc, Q = acc ^ 1u;
          mbar_wait(&bars->tmem_full[R], (eph >> R) & 1u);
          eph ^= 1u << R;
          const int nseg = (KB + SGT - 1) / SGT;
          for (int sg = 1; sg < nseg; ++sg) {
            mbar_wait(&bars->tmem_full[Q], (eph >> Q) & 1u);
            eph ^= 1u << Q;
            tc_fence_after();
#pragma unroll 1
            for (int c = (sub - ti * CHUNKS) & (EPI_SUBS - 1); c < CHUNKS; c += EPI_SUBS) {
              // all four loads of a chunk in flight together (the MMA stream waits for this region)
              uint32_t p0[16], q0[16], p1[16], q1[16];
              const uint32_t pa = tmem_base + lane_base + Q * BN + c * 32, qa = tmem_base + lane_base + R * BN + c * 32;
              tmem_ld_32x16(pa, p0);
              tmem_ld_32x16(qa, q0);
              tmem_ld_32x16(pa + 16, p1);
              tmem_ld_32x16(qa + 16, q1);
              tmem_ld_wait();
              if (c + EPI_SUBS >= CHUNKS) {
                // my last chunk of the partial is in registers: hand the region back before the add and the stores
                // (they touch the sum region only), ~150 cycles earlier on the MMA stream's critical path
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&bars->tmem_empty[Q]), 0));
              }
#pragma unroll
              for (int e = 0; e < 16; ++e) {
                q0[e] = __float_as_uint(__uint_as_float(q0[e]) + __uint_as_float(p0[e]));
                q1[e] = __float_as_uint(__uint_as_float(q1[e]) + __uint_as_float(p1[e]));
              }
              tmem_st_32x16(qa, q0);
              tmem_st_32x16(qa + 16, q1);
            }
            tmem_st_wait();
          }
        } else {
          mbar_wait(&bars->tmem_full[acc], acc_phase);
        }
        tc_fence_after();
        const uint32_t tmem_acc = tmem_base + lane_base + acc * BN;
        // every fourth chunk (counted over the whole row tile) is mine: start at it instead of testing each one
#pragma unroll 1
        for (int c = (sub - ti * CHUNKS) & (EPI_SUBS - 1); c < CHUNKS; c += EPI_SUBS) {
          uint32_t r[32];
          if (SEGM) {
            // my chunk of every partial accumulator of this tile, summed in fp32 registers; a partial buffer goes back
            // to the MMA stream as soon as it is read (the last one is released below like an ordinary accumulator)
            float sum[32];
            const int nseg = (KB + SEG - 1) / SEG;
            for (int seg = 0; seg < nseg; ++seg) {
              if (seg > 0) {
                mbar_wait(&bars->tmem_full[acc], acc_phase);
                tc_fence_after();
              }
              tmem_ld_32x32(tmem_base + lane_base + acc * BN + c * 32, r);
              tmem_ld_wait();
#pragma unroll
              for (int e = 0; e < 32; ++e) sum[e] = seg == 0 ? __uint_as_float(r[e]) : sum[e] + __uint_as_float(r[e]);
              if (seg < nseg - 1) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&bars->tmem_empty[acc]), 0));
                if (++acc == NACC) {
                  acc = 0;
                  acc_phase ^= 1;
                }
              }
            }
#pragma unroll
            for (int e = 0; e < 32; ++e) r[e] = __float_as_uint(sum[e]);
          } else {
            tmem_ld_32x32(tmem_acc + c * 32, r);
          }
          const int col = nt * BN + c * 32;
          const float4* wn4 = reinterpret_cast<const float4*>(wn_src + col);
          float4 w4[8];
          if (bias_mode) {  // wnorm is already in the accumulator
#pragma unroll
            for (int g = 0; g < 8; ++g) w4[g] = make_float4(0.f, 0.f, 0.f, 0.f);
          } else {
#pragma unroll
            for (int g = 0; g < 8; ++g) w4[g] = wn4[g];
          }
          tmem_ld_wait();
          if constexpr (NB > 2) {
            // top-k: my table keeps the k smallest (score, prototype) pairs of my chunks; `gate` is its k-th score.
            // Whatever does not enter (or leaves) lowers `evicted`; the row is flagged if that reaches the final bound.
            float sc[32];
            float c1 = kInf;
#pragma unroll
            for (int g = 0; g < 8; ++g) {
              sc[4 * g + 0] = fmaf(-2.f, __uint_as_float(r[4 * g + 0]), w4[g].x);
              sc[4 * g + 1] = fmaf(-2.f, __uint_as_float(r[4 * g + 1]), w4[g].y);
              sc[4 * g + 2] = fmaf(-2.f, __uint_as_float(r[4 * g + 2]), w4[g].z);
              sc[4 * g + 3] = fmaf(-2.f, __uint_as_float(r[4 * g + 3]), w4[g].w);
              c1 = fminf(c1, fminf(fminf(sc[4 * g + 0], sc[4 * g + 1]), fminf(sc[4 * g + 2], sc[4 * g + 3])));
            }
            if (c1 > gate) {  // the usual case once the table is full: one minimum
              evicted = fminf(evicted, c1);
              continue;
            }
            uint32_t need = 0;
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              const bool in = sc[e] <= gate;
              evicted = fminf(evicted, in ? __int_as_float(0x7f800000) : sc[e]);
              need |= (in ? 1u : 0u) << e;
            }
#pragma unroll 1
            while (need) {
              const int e = __ffs(need) - 1;
              need &= need - 1;
              const float se = sc[e];
              if (se > gate) {
                evicted = fminf(evicted, se);
              } else {
                const float2 o = slow_offer_topk(se, col + e, my_top_addr, epi_const_addr, n_topk);
                gate = o.x;
                evicted = fminf(evicted, o.y);
              }
            }
            continue;
          }
          // pass A: smallest score(s) of the chunk
          float a1 = kInf, a2 = kInf;
          float gm[8];  // minimum of each group of four columns: pass B re-examines only the groups in bound
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            const float s0 = fmaf(-2.f, __uint_as_float(r[4 * g + 0]), w4[g].x);
            const float s1 = fmaf(-2.f, __uint_as_float(r[4 * g + 1]), w4[g].y);
            const float s2 = fmaf(-2.f, __uint_as_float(r[4 * g + 2]), w4[g].z);
            const float s3 = fmaf(-2.f, __uint_as_float(r[4 * g + 3]), w4[g].w);
            gm[g] = fminf(fminf(s0, s1), fminf(s2, s3));
            if (NB == 2) {
              a2 = fminf(a2, fmaxf(a1, s0)); a1 = fminf(a1, s0);
              a2 = fminf(a2, fmaxf(a1, s1)); a1 = fminf(a1, s1);
              a2 = fminf(a2, fmaxf(a1, s2)); a1 = fminf(a1, s2);
              a2 = fminf(a2, fmaxf(a1, s3)); a1 = fminf(a1, s3);
            }
          }
          if (NB == 1) a1 = fminf(fminf(fminf(gm[0], gm[1]), fminf(gm[2], gm[3])), fminf(fminf(gm[4], gm[5]), fminf(gm[6], gm[7])));
          // fold into the running minima; NB == 1 also shares the minimum with the other three
          // warps of this row (a racy read-modify-write is fine: every value written is a score that
          // was really seen, so the threshold can only be looser than necessary, never tighter)
          if (TB) {
            // upper bounds: v of this chunk's best column; m1 / m2 = the two smallest of MY chunks (distinct columns, so
            // the merge below can form the second smallest upper bound of the row); the row shares its smallest one
            const float v = a1 + kb;
            const float sh = row_min[t];
            if (v < sh) row_min[t] = v;
            m2 = fminf(m2, fmaxf(m1, v));
            m1 = fminf(m1, v);
            thr = fminf(m1, sh) + kb;  // in score units for this tile: key <= U
          } else if (NB == 1) {
            const float sh = row_min[t];
            if (a1 < sh) row_min[t] = a1;
            m1 = fminf(m1, fminf(a1, sh));
            thr = m1 + tau;
          } else {
            m2 = fminf(fmaxf(m1, a1), fminf(m2, a2));
            m1 = fminf(m1, a1);
            thr = m2 < 1.0e38f ? m2 + tau : kInf;
          }
          // pass B on the live registers: offer what is inside the bound.  A score at or above the fast gate
          // cannot enter the table and only lowers `evicted`; the rest goes through slow_offer (one out-of-line
          // copy: the 16 epilogue warps share the instruction cache).  Three cases, cheapest first:
          //  * the whole chunk is at or above the gate (rows with thousands of near-identical prototypes inside
          //    their bound, once the table is full): one minimum;
          //  * exactly one score is in bound -- the chunk minimum itself, the usual "new running minimum" event:
          //    one call, made by all such lanes of the warp together;
          //  * several: the scores are parked in local memory so that a loop can index them, lanes advancing
          //    through their own in-bound scores in parallel.
          if (a1 <= thr) {
            if (a1 - kb >= gate) {
              evicted = fminf(evicted, a1 - kb);
            } else {
              uint32_t inb = 0;
#pragma unroll
              for (int g = 0; g < 8; ++g) {
                if (gm[g] <= thr) {  // usually one group per lane: the others cost a compare and a branch
                  inb |= (fmaf(-2.f, __uint_as_float(r[4 * g + 0]), w4[g].x) <= thr ? 1u : 0u) << (4 * g + 0);
                  inb |= (fmaf(-2.f, __uint_as_float(r[4 * g + 1]), w4[g].y) <= thr ? 1u : 0u) << (4 * g + 1);
                  inb |= (fmaf(-2.f, __uint_as_float(r[4 * g + 2]), w4[g].z) <= thr ? 1u : 0u) << (4 * g + 2);
                  inb |= (fmaf(-2.f, __uint_as_float(r[4 * g + 3]), w4[g].w) <= thr ? 1u : 0u) << (4 * g + 3);
                }
              }
              if ((inb & (inb - 1)) == 0) {
                if (inb) {
                  const float2 o = slow_offer(a1 - kb, col + __ffs(inb) - 1, my_val_addr, epi_const_addr);
                  gate = o.x;
                  evicted = fminf(evicted, o.y);
                }
              } else {
                float sc[32];
                uint32_t need = 0;
#pragma unroll
                for (int g = 0; g < 8; ++g) {
                  sc[4 * g + 0] = fmaf(-2.f, __uint_as_float(r[4 * g + 0]), w4[g].x);
                  sc[4 * g + 1] = fmaf(-2.f, __uint_as_float(r[4 * g + 1]), w4[g].y);
                  sc[4 * g + 2] = fmaf(-2.f, __uint_as_float(r[4 * g + 2]), w4[g].z);
                  sc[4 * g + 3] = fmaf(-2.f, __uint_as_float(r[4 * g + 3]), w4[g].w);
#pragma unroll
                  for (int e = 0; e < 4; ++e) {
                    // in bound but not below the gate as it stands (it only falls): evicted, branch-free
                    const float se = sc[4 * g + e];
                    const bool in = se <= thr, out = se - kb >= gate;
                    evicted = fminf(evicted, in && out ? se - kb : __int_as_float(0x7f800000));
                    need |= (in && !out ? 1u : 0u) << (4 * g + e);
                  }
                }
#pragma unroll 1
                while (need) {
                  const int e = __ffs(need) - 1;
                  need &= need - 1;
                  const float se = sc[e] - kb;
                  if (se >= gate) {
                    evicted = fminf(evicted, se);
                  } else {
                    const float2 o = slow_offer(se, col + e, my_val_addr, epi_const_addr);
                    gate = o.x;
                    evicted = fminf(evicted, o.y);
                  }
                }
              }
            }
          }
        }
        tc_fence_before();
        if (PAIR) {  // one arrive per warp, on the leader's barrier
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&bars->tmem_empty[acc]), 0));
        } else {
          mbar_arrive(&bars->tmem_empty[acc]);
        }
        if (++acc == NACC) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
      // merge the four trackers of each row
      sub_state[t * EPI_SUBS + sub] = make_float4(m1, m2, evicted, 0.f);
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS));
      if (sub == 0) {
        float g1 = kInf, g2 = kInf, ev = __int_as_float(0x7f800000);
#pragma unroll
        for (int q = 0; q < EPI_SUBS; ++q) {
          const float4 st = sub_state[t * EPI_SUBS + q];
          if (NB == 2 || TB) g2 = fminf(fmaxf(g1, st.x), fminf(g2, st.y));
          g1 = fminf(g1, st.x);
          ev = fminf(ev, st.z);
        }
        if constexpr (NB > 2) {
          // the k-th smallest score of the row: k steps of a merge of the four sorted tables (each holds its warp's k
          // smallest, so together they hold the row's k smallest); candidates = every kept pair within the bound of it
          const uint32_t tb = smem_u32(top_val + t);
          int h[EPI_SUBS] = {0, 0, 0, 0};
          float kth = kInf;
          for (int q = 0; q < n_topk; ++q) {
            float bv = __int_as_float(0x7f800000);
            int bj = 0x7fffffff, bs = 0;
#pragma unroll
            for (int u = 0; u < EPI_SUBS; ++u) {
              float v;
              int j;
              const uint32_t a = tb + (uint32_t)((u * KTOP + h[u]) * BM * 4);
              asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
              asm volatile("ld.shared.s32 %0, [%1];" : "=r"(j) : "r"(a + kTopIdxOffset));
              const bool take = pair_after(bv, bj, v, j);
              bv = take ? v : bv;
              bj = take ? j : bj;
              bs = take ? u : bs;
            }
#pragma unroll
            for (int u = 0; u < EPI_SUBS; ++u) h[u] += bs == u ? 1 : 0;
            kth = bv;
          }
          const float gthr = kth < 1.0e38f ? kth + tau : kInf;
          bool overflow = ev <= gthr;
          int cnt = 0;
          int32_t* slots = cand_idx + orow * kMaxCandK;
          for (int u = 0; u < EPI_SUBS; ++u) {
            for (int q = 0; q < n_topk; ++q) {  // sorted: the pairs in bound form a prefix
              float v;
              int j;
              const uint32_t a = tb + (uint32_t)((u * KTOP + q) * BM * 4);
              asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
              if (!(v <= gthr)) break;
              asm volatile("ld.shared.s32 %0, [%1];" : "=r"(j) : "r"(a + kTopIdxOffset));
              if (row < N && cnt < kMaxCandK) slots[cnt] = j;
              ++cnt;
            }
          }
          if (cnt > kMaxCandK) overflow = true;
          if (row < N) cand_count[orow] = (uint8_t)(overflow ? DBGSOM_CAND_OVERFLOW : cnt);
          row_min[t] = kInf;
        } else {
        const float gm = NB == 1 ? g1 : g2;
        // TB: the tables hold keys (score - tile bound) and g1 is the smallest upper bound: in bound iff key <= g1
        const float gthr = gm < 1.0e38f ? (TB ? gm : gm + tau) : kInf;
        // the sixteen (score, prototype) pairs of the row: independent loads first, then branch-free bookkeeping
        float v[EPI_SUBS * KSUB];
        int jx[EPI_SUBS * KSUB];
#pragma unroll
        for (int q = 0; q < EPI_SUBS; ++q) {
          const float4 v4 = lds_f4(smem_u32(tab_val + (t * EPI_SUBS + q) * KSUB));
          const int4 j4 = lds_i4(smem_u32(tab_idx + (t * EPI_SUBS + q) * KSUB));
          v[4 * q + 0] = v4.x; v[4 * q + 1] = v4.y; v[4 * q + 2] = v4.z; v[4 * q + 3] = v4.w;
          jx[4 * q + 0] = j4.x; jx[4 * q + 1] = j4.y; jx[4 * q + 2] = j4.z; jx[4 * q + 3] = j4.w;
        }
        int cnt = 0, best = -1;
        float bv = __int_as_float(0x7f800000), sv = __int_as_float(0x7f800000);  // two smallest scores kept
        bool overflow = ev <= gthr;
#pragma unroll
        for (int i = 0; i < EPI_SUBS * KSUB; ++i) {
          const bool in = v[i] <= gthr;  // free slots hold +inf, gthr is finite
          const bool first = in && (v[i] < bv || (v[i] == bv && jx[i] < best));
          const bool second = in && !first && v[i] < sv;
          cnt += in ? 1 : 0;
          sv = first ? bv : (second ? v[i] : sv);
          bv = first ? v[i] : bv;
          best = first ? jx[i] : best;
        }
        if (cnt > kMaxCand) overflow = true;
        if (row < N) {
          // candidate slots past the count are never read (bmu_resolve.cu); a row with one candidate -- almost all of
          // them -- writes one slot.  A flagged row has no candidate list; its first slot carries the gap between the
          // two smallest approximate scores instead (>= 0, float bits), which tightens the near-tie test of the re-score
          int32_t* slots = cand_idx + orow * kMaxCand;
          if (overflow) {
            // TB: second smallest upper bound minus smallest lower bound = a proven bound on the exact gap
            slots[0] = __float_as_int(fmaxf((TB ? (g2 < 1.0e38f ? g2 : __int_as_float(0x7f800000)) : sv) - bv, 0.f));
          } else if (cnt == 1) {
            slots[0] = best;
          } else {
            int w = 0;
#pragma unroll
            for (int i = 0; i < EPI_SUBS * KSUB; ++i)
              if (v[i] <= gthr) slots[w++] = jx[i];
          }
          cand_count[orow] = (uint8_t)(overflow ? DBGSOM_CAND_OVERFLOW : cnt);
          idx_out[orow * NB] = best;
        }
        row_min[t] = kInf;
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS));
    }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (CL > 1) cluster_sync_all();  // no CTA leaves while a peer may still write its shared memory or barriers
  if (warp == 2) {
    tc_fence_after();
    if (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)C::TMEM_COLS)
                   : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)C::TMEM_COLS)
                   : "memory");
  }
}

// ------------------------------------------------------------------------------------------ host
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// fp16 [rows, ld] row-major, box = 64 columns x box_rows, 128-byte swizzle, zero fill out of bounds
int make_map(CUtensorMap* map, const uint16_t* base, int64_t rows, int64_t ld, int box_rows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return DBGSOM_E_DRIVER;
  const cuuint64_t dims[2] = {(cuuint64_t)ld, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  const cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  const cuuint32_t elem[2] = {1, 1};
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<uint16_t*>(base), dims, strides, box, elem,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? DBGSOM_OK : DBGSOM_E_DRIVER;
}

int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

template <int NPASS, int NB, int BN, int RES_KB, int AKB, int CL, bool PAIR = false, int SEL = 0, bool TB = false, int SGT = 0>
int launch_cfg_cl(const dbgsom_bmu_args& a, const BmuWorkspace& ws, cudaStream_t s) {
  using C = Cfg<NPASS, BN, RES_KB, AKB, PAIR && AKB == 0 && RES_KB == 0, extra_bytes<NB, SEL>()>;
  CUtensorMap mxh, mxl, mwh, mwl;
  int rc = make_map(&mxh, a.d_X16_hi, a.N, a.ld16, BM);
  if (rc) return rc;
  rc = make_map(&mwh, a.d_W16_hi, a.Mpad, a.ld16, BN / CL);
  if (rc) return rc;
  if (NPASS == 3) {
    rc = make_map(&mxl, a.d_X16_lo, a.N, a.ld16, BM);
    if (rc) return rc;
    rc = make_map(&mwl, a.d_W16_lo, a.Mpad, a.ld16, BN / CL);
    if (rc) return rc;
  } else {
    mxl = mxh;
    mwl = mwh;
  }
  CUtensorMap mwb = mwh;
  // (the classic search, and the FLAG pass of the selective search for D <= 128, where its epilogue is the limiter)
  const bool with_bias = (SEL == 0 || (SEL == 1 && AKB <= 2)) && PAIR && C::ATM && a.d_Wb16 != nullptr && a.d_bias_scale != nullptr;
  if (with_bias) {
    rc = make_map(&mwb, a.d_Wb16, a.Mpad, BK, BN / CL);
    if (rc) return rc;
  }
  if (with_bias && getenv("DBGSOM_TC_VERBOSE")) {
    static bool said = false;
    if (!said) {
      said = true;
      float e = -1.f;
      cudaMemcpy(&e, a.d_bias_scale, sizeof(float), cudaMemcpyDeviceToHost);
      fprintf(stderr, "dbgsom: K1 takes wnorm through the bias k-step, E = %g\n", e);
    }
  }
  if (getenv("DBGSOM_TC_VERBOSE")) {  // once per process and kernel form (the static is per instantiation)
    static bool said = false;
    if (!said) {
      said = true;
      fprintf(stderr, "dbgsom: K1 form npass=%d nb=%d bn=%d res_kb=%d akb=%d cl=%d pair=%d sel=%d tb=%d sgt=%d\n", NPASS, NB,
              BN, RES_KB, AKB, CL, (int)PAIR, SEL, (int)TB, SGT);
    }
  }
  auto kern = bmu_cand_tensor_kernel<NPASS, NB, BN, RES_KB, AKB, CL, PAIR, SEL, TB, SGT>;
  DBGSOM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
  const int KB = (int)(a.ld16 / BK);
  const int NT = a.Mpad / BN;  // prototypes are permuted over all Mpad shadow rows
  int64_t grid = round_up<int64_t>(ceil_div<int64_t>(a.N, BM), CL);
  int64_t max_grid = sm_count() / CL * CL;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)max_grid);
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = C::SMEM_BYTES;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = CL > 1 ? 1 : 0;
  if (CL > 1) {  // persistent kernel: no more clusters than can be resident at once (GPC boundaries)
    static int max_clusters = 0;
    if (max_clusters == 0) {
      DBGSOM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 0));
      if (cudaOccupancyMaxActiveClusters(&max_clusters, kern, &cfg) != cudaSuccess || max_clusters <= 0) {
        (void)cudaGetLastError();
        max_clusters = sm_count() / CL;
      }
    }
    if (max_grid > (int64_t)max_clusters * CL) max_grid = (int64_t)max_clusters * CL;
  }
  if (grid > max_grid) grid = max_grid;
  cfg.gridDim = dim3((unsigned)grid);
  const float coef = tensor_bound_coef(NPASS, a.bound_scale);
  const float acc_coef = tensor_acc_coef_args(a);
  // the arithmetic form needs c * stride < 2^32 for every shadow row c
  const int pstride = a.proto_stride > 0 && a.Mpad <= 65535 && a.proto_stride < a.Mpad ? a.proto_stride : 0;
  DBGSOM_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, mxh, mxl, mwh, mwl, mwb, with_bias ? a.d_bias_scale : (const float*)nullptr,
                                     a.N, KB, NT, a.d_wnorm, a.d_proto_of_col, pstride,
                                     a.n_bmu == 1 ? a.ties_any : 0, a.d_xnorm16, a.d_wmax, coef, acc_coef, a.d_idx, ws.cand_idx, ws.cand_count,
                                     a.d_row_perm, reinterpret_cast<unsigned long long*>(a.d_tile_mask),
                                     a.select_granule == 64 ? 6 : 7,
                                     a.d_stats ? reinterpret_cast<unsigned long long*>(a.d_stats) + 4 : (unsigned long long*)nullptr,
                                     TB ? a.d_tile_bound : (const float*)nullptr, a.n_bmu));
  DBGSOM_LAUNCH_CHECK();
  return DBGSOM_OK;
}

// cluster size: 2 by default (prototype tiles multicast to a CTA pair); DBGSOM_TC_CLUSTER = 1 | 2 | 4 overrides
int cluster_size() {
  static int cl = 0;
  if (cl == 0) {
    const char* e = getenv("DBGSOM_TC_CLUSTER");
    cl = e ? atoi(e) : 2;
    if (cl != 1 && cl != 2 && cl != 4) cl = 2;
  }
  return cl;
}

template <int NPASS, int NB, int BN, int RES_KB, int AKB = 0>
int launch_cfg(const dbgsom_bmu_args& a, const BmuWorkspace& ws, cudaStream_t s) {
  // small problems (fewer row tiles than SMs) gain nothing from sharing
  const int cl = ceil_div<int64_t>(a.N, BM) < sm_count() ? 1 : cluster_size();
  if constexpr (AKB > 0) {  // CTA pairs (cta_group::2) whenever the sample tile is tensor-memory resident; DBGSOM_TC_PAIR=0 disables
    static const bool pair = getenv("DBGSOM_TC_PAIR") == nullptr || atoi(getenv("DBGSOM_TC_PAIR")) != 0;
    if (pair && cl >= 2) return launch_cfg_cl<NPASS, NB, BN, RES_KB, AKB, 2, true>(a, ws, s);
  }
  if (cl == 4) return launch_cfg_cl<NPASS, NB, BN, RES_KB, AKB, 4>(a, ws, s);
  if (cl == 2) return launch_cfg_cl<NPASS, NB, BN, RES_KB, AKB, 2>(a, ws, s);
  return launch_cfg_cl<NPASS, NB, BN, RES_KB, AKB, 1>(a, ws, s);
}

// which form runs for D > 256 (three passes): the decisions are functions of the arguments so that the re-score
// (bmu_resolve.cu) can use the error bound of the form that produced the candidates
bool streamed_pairs(const dbgsom_bmu_args& a) {
  static const bool pairs = getenv("DBGSOM_TC_PAIR") == nullptr || atoi(getenv("DBGSOM_TC_PAIR")) != 0;
  return a.backend == DBGSOM_BMU_TENSOR && a.n_pass == 3 && a.ld16 / BK > MAX_RES_KB && pairs && cluster_size() >= 2 &&
         ceil_div<int64_t>(a.N, BM) >= sm_count();
}
// DBGSOM_TC_SEGM: 3 (default) / 2 = segmented accumulation with 256-column MMAs and the running sums in tensor memory,
// chains of 4 / 8 k-blocks; 1 = segmented accumulation with 128-column MMAs, running sums in registers (the first
// segmented form: same bound as 3, but HBM bound on re-streamed sample tiles); 0 = one chain, 256-column MMAs.
// Config-5 shard (625k x 4096 rows, 16384 prototypes), candidate search per epoch: 221 / 212 / 289 / 193 ms.
int streamed_segm_mode() {
  static const int mode = getenv("DBGSOM_TC_SEGM") == nullptr ? 3 : atoi(getenv("DBGSOM_TC_SEGM"));
  return mode;
}
bool streamed_segmented(const dbgsom_bmu_args& a) { return streamed_segm_mode() == 1 && streamed_pairs(a); }
int streamed_tmem_sums(const dbgsom_bmu_args& a) {  // k-blocks per chain, 0 = another form
  const int mode = streamed_segm_mode();
  return (mode == 2 || mode == 3) && streamed_pairs(a) ? (mode == 2 ? 8 : 4) : 0;
}
}  // namespace
// per-tile error bounds (template flag TB): the streamed pair forms, one winner, the caller supplied the tile maxima
bool tile_bounds_active(const dbgsom_bmu_args& a) {
  return a.d_tile_bound != nullptr && a.n_bmu == 1 && a.select == DBGSOM_SELECT_OFF && streamed_pairs(a);
}
namespace {

template <int NPASS, int NB>
int launch_shape(const dbgsom_bmu_args& a, const BmuWorkspace& ws, cudaStream_t s) {
  // Tile shapes by shared-memory budget (227 KB): the resident sample tile takes 16 KB per k-block
  // (x2 with the lo shadow); what is left must hold >= 4 stages of prototypes to cover TMA latency.
  const int KB = (int)(a.ld16 / BK);
  if constexpr (NPASS == 1) {
    if (KB <= 2) return launch_cfg<NPASS, NB, 256, 2>(a, ws, s);
    if (KB <= MAX_RES_KB) return launch_cfg<NPASS, NB, 256, 4>(a, ws, s);
    return launch_cfg<NPASS, NB, 256, 0>(a, ws, s);
  } else {
    static const bool a_smem = getenv("DBGSOM_TC_A_SMEM") != nullptr;  // tuning switch: sample tile in smem
    if constexpr (NB > 2) {  // the top-k tables leave no room for a resident sample tile in shared memory
      if (KB <= 2) return launch_cfg<NPASS, NB, 128, 0, 2>(a, ws, s);
      if (KB <= MAX_RES_KB) return launch_cfg<NPASS, NB, 128, 0, 4>(a, ws, s);
    } else {
      if (KB <= 2) return a_smem ? launch_cfg<NPASS, NB, 128, 2>(a, ws, s) : launch_cfg<NPASS, NB, 128, 0, 2>(a, ws, s);
      if (KB <= MAX_RES_KB)
        return a_smem ? launch_cfg<NPASS, NB, 128, 4>(a, ws, s) : launch_cfg<NPASS, NB, 128, 0, 4>(a, ws, s);
    }
    // D > 256: both operands stream.  As CTA pairs with 256-column MMAs each CTA stages its 128 sample rows and HALF
    // of a 256-prototype tile per k-block (the single-CTA form wants 208 B/clk from the shared-memory pipe, this 104)
    if (streamed_pairs(a)) {
      // segmented accumulation (chains of four k-blocks; 256-column tiles with the running sums in tensor memory, or
      // 128-column tiles with the sums in registers) keeps the error bound of D = 256 at any D; DBGSOM_TC_SEGM=0
      // selects the one-chain form with 256-column tiles
      const int sgt = streamed_tmem_sums(a);
      if constexpr (NB == 1) {
        if (tile_bounds_active(a)) {
          if (streamed_segmented(a)) return launch_cfg_cl<NPASS, NB, 128, 0, 0, 2, true, 0, true>(a, ws, s);
          if (sgt == 8) return launch_cfg_cl<NPASS, NB, 256, 0, 0, 2, true, 0, true, 8>(a, ws, s);
          if (sgt == 4) return launch_cfg_cl<NPASS, NB, 256, 0, 0, 2, true, 0, true, 4>(a, ws, s);
          return launch_cfg_cl<NPASS, NB, 256, 0, 0, 2, true, 0, true>(a, ws, s);
        }
      }
      if (streamed_segmented(a)) return launch_cfg_cl<NPASS, NB, 128, 0, 0, 2, true>(a, ws, s);
      if (sgt == 8) return launch_cfg_cl<NPASS, NB, 256, 0, 0, 2, true, 0, false, 8>(a, ws, s);
      if (sgt == 4) return launch_cfg_cl<NPASS, NB, 256, 0, 0, 2, true, 0, false, 4>(a, ws, s);
      return launch_cfg_cl<NPASS, NB, 256, 0, 0, 2, true>(a, ws, s);
    }
    return launch_cfg<NPASS, NB, 128, 0>(a, ws, s);
  }
}

}  // namespace

float tensor_acc_coef_args(const dbgsom_bmu_args& a) {
  if (streamed_segmented(a)) {  // chains of 48 steps like D = 256, plus the fp32 sums of the partial tiles
    double c = 2.4e-7 * (a.strict ? 4.0 : 2.0);
    if (const char* e = getenv("DBGSOM_ACC_SCALE")) c *= atof(e);
    return (float)c;
  }
  if (const int sgt = streamed_tmem_sums(a)) {  // chains of 12 * sgt steps (48 at four k-blocks), plus the fp32 sums
    const double grow = (double)sgt / 4.0;
    double c = 2.4e-7 * (a.strict ? 4.0 * grow : 2.0 * sqrt(grow));
    if (const char* e = getenv("DBGSOM_ACC_SCALE")) c *= atof(e);
    return (float)c;
  }
  return tensor_acc_coef(a.n_pass, a.ld16, a.strict);
}

bool bmu_select_supported(int64_t N, int64_t ld16, int Mpad, int n_bmu, int granule) {
  if (n_bmu != 1 || (granule != 64 && granule != 128)) return false;
  if (ld16 % BK != 0 || ld16 / BK > MAX_RES_KB || ld16 / BK < 1) return false;  // sample tile in tensor memory: D <= 256
  if (Mpad % 256 != 0 || Mpad / granule > 64 || Mpad > kFlagMaxCols) return false;  // one mask bit per column tile
  if (ceil_div<int64_t>(N, BM) < sm_count()) return false;                        // CTA pairs need a full wave of row tiles
  return cluster_size() >= 2;
}

namespace {
template <int SEL>
int launch_select(const dbgsom_bmu_args& a, const BmuWorkspace& ws, cudaStream_t s) {
  const int KB = (int)(a.ld16 / BK);
  if constexpr (SEL == 1) {  // FLAG: one pass, 128-column MMAs
    if (KB <= 2) return launch_cfg_cl<1, 1, 128, 0, 2, 2, true, 1>(a, ws, s);
    return launch_cfg_cl<1, 1, 128, 0, 4, 2, true, 1>(a, ws, s);
  } else {                   // REFINE: three passes over the flagged column tiles of `select_granule` prototypes
    if (a.select_granule == 64) {
      if (KB <= 2) return launch_cfg_cl<3, 1, 64, 0, 2, 2, true, 2>(a, ws, s);
      return launch_cfg_cl<3, 1, 64, 0, 4, 2, true, 2>(a, ws, s);
    }
    if (KB <= 2) return launch_cfg_cl<3, 1, 128, 0, 2, 2, true, 2>(a, ws, s);
    return launch_cfg_cl<3, 1, 128, 0, 4, 2, true, 2>(a, ws, s);
  }
}
}  // namespace

int launch_bmu_cand_tensor(const dbgsom_bmu_args& a, const BmuWorkspace& ws, cudaStream_t s) {
  if (a.ld16 % BK != 0 || a.Mpad % 256 != 0 || a.Mpad < a.M) return DBGSOM_E_UNSUPPORTED;
  if (a.select != DBGSOM_SELECT_OFF) {
    if (!bmu_select_supported(a.N, a.ld16, a.Mpad, a.n_bmu, a.select_granule) || !a.d_proto_of_col) return DBGSOM_E_UNSUPPORTED;
    if (a.N > 0x7fffff00LL) return DBGSOM_E_UNSUPPORTED;
    return a.select == DBGSOM_SELECT_FLAG ? launch_select<1>(a, ws, s) : launch_select<2>(a, ws, s);
  }
  if (!a.d_proto_of_col) return DBGSOM_E_BADARG;
  if ((reinterpret_cast<uintptr_t>(a.d_X16_hi) & 15u) || (reinterpret_cast<uintptr_t>(a.d_W16_hi) & 15u) ||
      (reinterpret_cast<uintptr_t>(a.d_wnorm) & 15u))
    return DBGSOM_E_UNSUPPORTED;
  if (a.N > 0x7fffff00LL) return DBGSOM_E_UNSUPPORTED;  // TMA coordinates are int32
  if (a.n_bmu > 2) return a.n_pass == 3 ? launch_shape<3, KTOP>(a, ws, s) : DBGSOM_E_UNSUPPORTED;
  if (a.n_pass == 1) return a.n_bmu == 1 ? launch_shape<1, 1>(a, ws, s) : launch_shape<1, 2>(a, ws, s);
  return a.n_bmu == 1 ? launch_shape<3, 1>(a, ws, s) : launch_shape<3, 2>(a, ws, s);
}

}  // namespace dbgsom
