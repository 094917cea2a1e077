// K2: sample weights + per-BMU segmented accumulation (HBM-bound; reads X exactly once).
//
// Replaces, per epoch (dbgsom/BaseSom.py):
//   _calculate_exp_similarity                      :533-538   k_i = 1 - sqrt(1 - exp(-d_i^2 / V))  (float64)
//   np.argsort(winners) / np.unique(return_index)  :488-489   -> counting sort by winner
//   numba_voronoi_set_centers                      :1028-1055 -> Sk_j = sum k_i x_i, sk_j = sum k_i
//   neuron_activations                             :500-503   -> n_j
//   numba_quantization_error                       :1058-1073 -> E_j = sum d_i
//
// Pipeline (all on one stream):
//   histogram (counts per winner [+ class histogram]) -> exclusive scan (segment offsets, n_j as
//   float64) -> scatter (sample permutation grouped by winner) -> segmented accumulate.
// The accumulate kernel gives every team of warps one contiguous range of the permutation; the
// team keeps the current segment's float64 prototype in registers (so the exact distance
// ||x_i - w_b|| costs no extra memory traffic), accumulates k_i x_i in float64 registers and
// flushes whenever the segment changes: the segment's first team stores its sums, teams that
// continue it leave theirs to acc_cont_kernel, which adds them in team order.  With the stable
// permutation every sum is taken in the same order on every run, so the result is bitwise
// repeatable (the fit is chaotic where prototypes collapse: a last-bit difference flips a near-tie
// winner and grows from there).  Everything after the fp32 load of x is float64 and matches the
// reference to ~1e-13; its convergence test (sum ||dW|| < 1e-5,
// dbgsom/BaseSom.py:519-522) needs that: with fp32 weights or partial sums the prototypes jitter
// by ~1e-7 relative from epoch to epoch and the fit stops at a different epoch (or never).
// B200 has the float64 rate for this (~3 DFMA per sample element, far below the HBM time).  The M x D table is never privatised in
// shared memory (4 MB at 4096 x 256); traffic is N*(4D+8) + a few M*D words.
#include <cstdlib>
#include <type_traits>

#include "common.cuh"

namespace dbgsom {

namespace {

// ------------------------------------------------------------------------------------------ histogram
constexpr int HIST_THREADS = 256;
constexpr int HIST_SMEM_BINS = 8192;

// counts[b] (and class_hist[b, y]) via shared-memory privatisation when the bin count is small
// (few bins => heavy contention on global atomics), plain global atomics otherwise.
template <bool SMEM>
__global__ void __launch_bounds__(HIST_THREADS) hist_kernel(const int32_t* __restrict__ bmu, int64_t N, int M,
                                                           const int32_t* __restrict__ labels, int n_classes,
                                                           int32_t* __restrict__ counts,
                                                           int32_t* __restrict__ class_hist, int64_t rows_per_block) {
  extern __shared__ int32_t sh[];
  const int nbins_c = labels ? M * n_classes : 0;
  if (SMEM) {
    for (int i = threadIdx.x; i < M + nbins_c; i += HIST_THREADS) sh[i] = 0;
    __syncthreads();
  }
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r1 = r0 + rows_per_block < N ? r0 + rows_per_block : N;
  for (int64_t i = r0 + threadIdx.x; i < r1; i += HIST_THREADS) {
    const int b = bmu[i];
    if ((unsigned)b >= (unsigned)M) continue;  // defensive: a NaN row has no winner
    if (SMEM) {
      atomicAdd(&sh[b], 1);
      if (labels) atomicAdd(&sh[M + b * n_classes + labels[i]], 1);
    } else {
      atomicAdd(&counts[b], 1);
      if (labels) atomicAdd(&class_hist[(int64_t)b * n_classes + labels[i]], 1);
    }
  }
  if (SMEM) {
    __syncthreads();
    for (int i = threadIdx.x; i < M; i += HIST_THREADS)
      if (sh[i]) atomicAdd(&counts[i], sh[i]);
    for (int i = threadIdx.x; i < nbins_c; i += HIST_THREADS)
      if (sh[M + i]) atomicAdd(&class_hist[i], sh[M + i]);
  }
}

// ------------------------------------------------------------------------------------------ scan
// single CTA: offsets[j] = sum_{i<j} counts[i], offsets[M] = total; n_j -> part_n (if given) as float64; cursor = 0
constexpr int SCAN_THREADS = 1024;
__global__ void __launch_bounds__(SCAN_THREADS) scan_kernel(const int32_t* __restrict__ counts, int M,
                                                           int32_t* __restrict__ offsets,
                                                           int32_t* __restrict__ cursor, double* __restrict__ part_n) {
  __shared__ int32_t warp_tot[32];
  __shared__ int32_t carry_sh;
  if (threadIdx.x == 0) carry_sh = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int base = 0; base < M; base += SCAN_THREADS) {
    const int j = base + threadIdx.x;
    const int32_t c = j < M ? counts[j] : 0;
    int32_t v = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int32_t t = __shfl_up_sync(kFullMask, v, o);
      if (lane >= o) v += t;
    }
    if (lane == 31) warp_tot[warp] = v;
    __syncthreads();
    if (warp == 0) {
      int32_t t = warp_tot[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int32_t u = __shfl_up_sync(kFullMask, t, o);
        if (lane >= o) t += u;
      }
      warp_tot[lane] = t;  // inclusive totals of warps
    }
    __syncthreads();
    const int32_t carry = carry_sh;
    const int32_t excl = carry + (warp ? warp_tot[warp - 1] : 0) + v - c;
    if (j < M) {
      offsets[j] = excl;
      cursor[j] = 0;
      if (part_n) part_n[j] = (double)c;
    }
    __syncthreads();
    if (threadIdx.x == SCAN_THREADS - 1) carry_sh = carry + warp_tot[31];
    __syncthreads();
  }
  if (threadIdx.x == 0) offsets[M] = carry_sh;
}

// ------------------------------------------------------------------------------------------ scatter
// perm[offsets[b] + slot] = i, slots handed out per winner; lanes of a warp that share a winner
// take consecutive slots from one atomic (few prototypes => thousands of samples per address).
constexpr int SCAT_THREADS = 256;
__global__ void __launch_bounds__(SCAT_THREADS) scatter_kernel(const int32_t* __restrict__ bmu, int64_t N, int M,
                                                              const int32_t* __restrict__ offsets,
                                                              int32_t* __restrict__ cursor, int32_t* __restrict__ perm) {
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * SCAT_THREADS;
  const int64_t n_round = round_up<int64_t>(N, 32);
  for (int64_t i = (int64_t)blockIdx.x * SCAT_THREADS + threadIdx.x; i < n_round; i += stride) {
    int b = i < N ? bmu[i] : -1;
    if ((unsigned)b >= (unsigned)M) b = -1;
    const unsigned peers = __match_any_sync(kFullMask, b);
    const int leader = __ffs(peers) - 1;
    const int rank = __popc(peers & ((1u << lane) - 1));
    int base = 0;
    if (lane == leader && b >= 0) base = atomicAdd(&cursor[b], __popc(peers));
    base = __shfl_sync(kFullMask, base, leader);
    if (b >= 0) perm[offsets[b] + base + rank] = (int32_t)i;
  }
}

// Stable counting sort for maps of up to STABLE_MAX_M neurons: perm lists the samples of each winner in
// ascending sample index, so the order K2 sums in -- and the sample order the selective search rebuilds its
// shadows in -- is the same on every run.  Each warp owns one contiguous chunk of samples:
//   stable_count_kernel  T[c][j] = samples of chunk c won by j (per-warp table in shared memory);
//   stable_base_kernel   T[c][j] = offsets[j] + sum_{c' < c} T[c'][j] (in place, one column per thread);
//   stable_place_kernel  the warp walks its chunk in index order, 32 samples at a time, and hands out the
//                        slots of its run per winner (lanes that share a winner: in lane order).
constexpr int STABLE_MAX_M = 24576;
constexpr int STABLE_MAX_CHUNKS = 148 * 8;
constexpr int STABLE_SMEM = 64 * 1024;  // per CTA: warps * M counters
constexpr int STABLE_PREFETCH = 8;      // 32-sample groups loaded ahead by the placing warp

struct StableChunks {
  int64_t chunk, n;  // samples per warp, number of warps (chunks)
  int warps;         // warps per CTA
};
__host__ __device__ inline int64_t stable_max_chunks(int64_t N) {
  const int64_t c = (N + 2047) / 2048;
  return c < 1 ? 1 : (c > STABLE_MAX_CHUNKS ? STABLE_MAX_CHUNKS : c);
}
inline StableChunks stable_chunks(int64_t N, int M) {
  StableChunks s;
  const int64_t want = stable_max_chunks(N);
  s.chunk = round_up<int64_t>(ceil_div<int64_t>(N, want), 32 * STABLE_PREFETCH);
  s.n = ceil_div<int64_t>(N, s.chunk);
  if (s.n < 1) s.n = 1;
  int w = STABLE_SMEM / (M * 4);
  s.warps = w < 1 ? 1 : (w > 8 ? 8 : w);
  return s;
}

__global__ void stable_count_kernel(const int32_t* __restrict__ bmu, int64_t N, int M, int64_t chunk, int64_t n_chunks,
                                    int32_t* __restrict__ T) {
  extern __shared__ int32_t st_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t c = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
  if (c >= n_chunks) return;
  int32_t* cnt = st_smem + (size_t)warp * M;
  for (int j = lane; j < M; j += 32) cnt[j] = 0;
  __syncwarp();
  const int64_t c0 = c * chunk, c1 = c0 + chunk < N ? c0 + chunk : N;
  for (int64_t i = c0 + lane; i < c1; i += 32) {
    const int b = bmu[i];
    if ((unsigned)b < (unsigned)M) atomicAdd(&cnt[b], 1);
  }
  __syncwarp();
  for (int j = lane; j < M; j += 32) T[c * M + j] = cnt[j];
}

__global__ void __launch_bounds__(1024) stable_base_kernel(int32_t* __restrict__ T, int64_t n_chunks, int M,
                                                          const int32_t* __restrict__ offsets) {
  __shared__ int32_t tot[32][33];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + lane;
  const int64_t r0 = n_chunks * w / 32, r1 = n_chunks * (w + 1) / 32;
  int32_t s = 0;
  if (j < M)
    for (int64_t r = r0; r < r1; ++r) s += T[r * M + j];
  tot[w][lane] = s;
  __syncthreads();
  if (j < M) {
    int32_t run = offsets[j];
    for (int q = 0; q < w; ++q) run += tot[q][lane];
    for (int64_t r = r0; r < r1; ++r) {
      const int32_t c = T[r * M + j];
      T[r * M + j] = run;
      run += c;
    }
  }
}

__global__ void stable_place_kernel(const int32_t* __restrict__ bmu, int64_t N, int M, int64_t chunk, int64_t n_chunks,
                                    const int32_t* __restrict__ T, int32_t* __restrict__ perm) {
  extern __shared__ int32_t st_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t c = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
  if (c >= n_chunks) return;
  int32_t* base = st_smem + (size_t)warp * M;
  for (int j = lane; j < M; j += 32) base[j] = T[c * M + j];
  __syncwarp();
  const int64_t c0 = c * chunk, c1 = c0 + chunk < N ? c0 + chunk : N;
  const unsigned lt = (1u << lane) - 1u;
  for (int64_t s = c0; s < c1; s += 32 * STABLE_PREFETCH) {
    int bb[STABLE_PREFETCH];
#pragma unroll
    for (int k = 0; k < STABLE_PREFETCH; ++k) {
      const int64_t i = s + k * 32 + lane;
      bb[k] = i < c1 ? bmu[i] : -1;
    }
#pragma unroll
    for (int k = 0; k < STABLE_PREFETCH; ++k) {
      const int b = (unsigned)bb[k] < (unsigned)M ? bb[k] : -1;
      const unsigned peers = __match_any_sync(kFullMask, b);
      const int leader = __ffs(peers) - 1;
      int pos = 0;
      if (b >= 0 && lane == leader) {
        pos = base[b];
        base[b] = pos + __popc(peers);
      }
      pos = __shfl_sync(kFullMask, pos, leader);
      if (b >= 0) perm[pos + __popc(peers & lt)] = (int32_t)(s + k * 32 + lane);
      __syncwarp();
    }
  }
}

// ------------------------------------------------------------------------------------------ accumulate
constexpr int ACC_WIN_BYTES = (64 + 8) * 8 + 64;  // row-offset ring of a warp (+ mirror), padded to 640 bytes
__device__ __forceinline__ uint32_t acc_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// float -> double without the XU pipe.  ncu showed the first version of this kernel bound by
// F2F.F64.F32 (sm__inst_executed_pipe_xu at 109 % of peak: ~4 conversions per clock and SM); the
// same value comes from four integer operations on the ALU/FMA pipes: the float's
// exponent/mantissa field shifted right by 3 plus the bias difference (1023 - 127) << 20.  Exact
// for normal floats; zeros and denormals come out with magnitude < 1.2e-38 instead of exactly
// themselves, far below anything a float64 sum of the data can resolve; inputs are finite
// (check_array), so the inf/NaN encodings never occur.
__device__ __forceinline__ double f32_as_f64(float f) {
  const uint32_t b = __float_as_uint(f);
  const uint32_t t = b & 0x7fffffffu;
  const uint32_t hi = (__umulhi(t, 0x20000000u) + 0x38000000u) | (b & 0x80000000u);
  return __hiloint2double((int)hi, (int)(b << 29));
}

// VPL : float4 per lane per row slab;  WPR : warps cooperating on one row (team size);
// U   : rows per batch (their sample weights are evaluated together, lane group u doing row u, so
//       the float64 exp/sqrt costs 1/U per row);  STAGES : depth of the copy ring.
// Every team owns one contiguous range of the sorted sequence; warp tw of a team handles columns
// [tw * 128 * VPL, (tw + 1) * 128 * VPL) of each row, and every LANE stages exactly the 16-byte
// pieces it consumes itself: HBM -> shared memory with cp.async (LDGSTS, L2 only), one commit group
// per batch, STAGES - 1 batches in flight per warp.  Shared memory is therefore a private staging
// area per lane -- no barrier, fence or elected issuer is involved and no registers are tied up by
// loads in flight.  (The second version used one bulk copy per row issued by an elected lane:
// ~30 instructions per copy on the uniform datapath, 18 % of the kernel's instruction stream.)
// Each element is converted to float64 ONCE and stays in registers (U * VPL * 4 doubles per lane) for
// both uses -- the distance and, once the row's weight is known, the k * x sum: the first version
// converted twice and was issue bound on the conversions (ncu: 69 % of the issue slots, 42 % of
// DRAM peak).
// Loop control (fourth version): the prefetch side owns the only cursor into the segment table.  It turns the
// permutation into BYTE OFFSETS of the rows, 32 positions at a time (one coalesced load, fetched one window
// ahead), in a 64-slot ring in shared memory, so that a row of a batch costs one broadcast ld.shared.u64 + one
// 64-bit add + the copies; the rows-per-batch decision (never across a segment boundary) travels to the consuming
// side through a byte FIFO in a register (bit 7 = "first batch of a segment").  The third version evaluated the
// segment cursor twice and selected each row index with two shuffles out of a register window: ~160 of the 519
// instructions per 4-row batch were loop control.
// All arithmetic is float64: distances by direct differences, k = 1 - sqrt(1 - exp(-d^2 / V))
// literally as dbgsom/BaseSom.py:536-537, sums in float64 registers.
// WGT (frequency weights, `weight` [N] float64): row i counts w_i times -- k_i, d_i and the count 1 of the row are
// multiplied by w_i, and the segment's weight sum is flushed into the n slot of `part` (the scan's integer count is
// overwritten).  Lane u of the issuing warp copies the weight of row u of the batch next to the staged rows, so the
// weight arrives with the batch's commit group; its sample index is the ring's byte offset / row bytes (exact in
// float64 for any N that fits the int32 permutation).
template <int VPL, int WPR, int U, int THREADS, int STAGES, bool FULLD, int XU, bool WGT>
__global__ void __launch_bounds__(THREADS, 2) accumulate_kernel(
    const float* __restrict__ X, int64_t N, int D, int64_t ldx, const int32_t* __restrict__ perm,
    const int32_t* __restrict__ offsets, const double* __restrict__ W, int M, double inv_var,
    const double* __restrict__ weight, double* __restrict__ part, double* __restrict__ cont,
    int32_t* __restrict__ cont_seg) {
  constexpr int TEAMS = THREADS / 32 / WPR;
  constexpr int SLOT_BYTES = U * VPL * 512;          // one batch of one warp
  constexpr int WGT_BYTES = WGT ? STAGES * U * 8 : 0;
  constexpr int WARP_BYTES = STAGES * SLOT_BYTES + VPL * 1024 + ACC_WIN_BYTES + WGT_BYTES;
  constexpr int CW = WGT ? 3 : 2;                    // sums per segment besides Sk in a continuation partial
  // per warp: [STAGES][U][VPL][32 lanes x 16 B] staged samples, then [VPL][32 lanes x 32 B] the current
  // segment's float64 prototype (each lane keeps the 4 columns it owns; in registers it cost 16 of them),
  // then the ring of row offsets: slot (p & 63) = byte offset of the row at position p; slots 0..7 are
  // mirrored at 64..71 so a batch reads its <= 8 consecutive slots without wrapping; WGT: then [STAGES][U]
  // float64 row weights
  static_assert(U <= 8 && STAGES >= 2 && STAGES <= 4, "offset ring mirror / byte FIFO");
  extern __shared__ __align__(16) uint8_t stage_smem[];
  __shared__ double red[TEAMS][2][WPR][U];  // cross-warp partial squared distances (double buffered)

  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int team = warp / WPR;
  const int tw = warp % WPR;
  const int col0 = tw * 128 * VPL + lane * 4;
  const int32_t total = offsets[M];  // samples that have a winner (== N without NaN rows)
  const uint32_t my_smem = acc_smem_u32(stage_smem) + (uint32_t)warp * WARP_BYTES + lane * 16;
  constexpr uint32_t W_OFF = STAGES * SLOT_BYTES;  // prototype area relative to my_smem: [VPL][2 halves][32 lanes x 16 B]
  bool act[VPL];  // FULLD: D == 128 * VPL * WPR, every slab of every lane is inside the row
#pragma unroll
  for (int v = 0; v < VPL; ++v) act[v] = FULLD || col0 + v * 128 < D;

  const int64_t n_teams = (int64_t)gridDim.x * TEAMS;
  const int64_t team_id = (int64_t)blockIdx.x * TEAMS + team;
  const int32_t p_begin = (int32_t)((int64_t)total * team_id / n_teams);
  const int32_t p_end = (int32_t)((int64_t)total * (team_id + 1) / n_teams);
  if (p_begin >= p_end) return;  // whole team exits together (no block-wide barrier follows)

  // segment containing p_begin: largest j with offsets[j] <= p_begin
  int lo = 0, hi = M;  // invariant offsets[lo] <= p_begin < offsets[hi]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (offsets[mid] <= p_begin) lo = mid; else hi = mid;
  }
  // prefetch side: next position, its segment and the segment's end; offset ring filled up to `filled`
  int32_t pp = p_begin, pseg = lo, pseg_end = offsets[lo + 1];
  bool pnew = true;  // the next batch is the first one this team takes from its segment
  int32_t filled = p_begin;
  const uint32_t my_win = acc_smem_u32(stage_smem) + (uint32_t)warp * WARP_BYTES + STAGES * SLOT_BYTES + VPL * 1024;
  auto perm_at = [&](int32_t p) { return perm[p < p_end ? p : p_end - 1]; };  // positions past the range are never used
  int32_t perm_nxt = perm_at(filled + lane);  // always one window ahead of the ring
  const uint32_t row_bytes = (uint32_t)ldx * 4u;
  const char* __restrict__ my_src = reinterpret_cast<const char*>(X + col0);
  const uint32_t my_wgt = my_win + ACC_WIN_BYTES;  // WGT: [STAGES][U] weights of the staged rows
  const double inv_row_bytes = 1.0 / (double)row_bytes;
  uint32_t fifo = 0;  // one byte per batch in flight, oldest lowest: rows | 0x80 if the batch starts a segment

  auto issue = [&](int stage, int fifo_pos) {  // every lane copies its own 16-byte pieces of the next batch
    if (pp < p_end) {
      while (pp >= pseg_end) {  // skip empty segments
        ++pseg;
        pseg_end = offsets[pseg + 1];
        pnew = true;
      }
      const int32_t lim = p_end < pseg_end ? p_end : pseg_end;
      const int nb = lim - pp < U ? lim - pp : U;
      if (pp + U > filled) {  // next 32 positions into the ring (never over a slot that is still to be read)
        const uint32_t slot = (uint32_t)(filled + lane) & 63u;
        const uint64_t off = (uint64_t)(uint32_t)perm_nxt * row_bytes;
        asm volatile("st.shared.u64 [%0], %1;" ::"r"(my_win + slot * 8), "l"(off) : "memory");
        if (slot < 8) asm volatile("st.shared.u64 [%0], %1;" ::"r"(my_win + (slot + 64) * 8), "l"(off) : "memory");
        filled += 32;
        perm_nxt = perm_at(filled + lane);
        __syncwarp();
      }
      const uint32_t wa = my_win + (((uint32_t)pp & 63u) << 3);
      const uint32_t dst = my_smem + (uint32_t)stage * SLOT_BYTES;
      uint64_t off[U];  // all U slots are read (the mirror keeps them inside the ring), only nb rows are copied
#pragma unroll
      for (int u = 0; u < U; ++u) asm volatile("ld.shared.u64 %0, [%1];" : "=l"(off[u]) : "r"(wa + u * 8));
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (u < nb) {
          const char* src = my_src + off[u];
#pragma unroll
          for (int v = 0; v < VPL; ++v)
            if (FULLD || act[v])
              asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + (u * VPL + v) * 512),
                           "l"(src + v * 512)
                           : "memory");
        }
      }
      if constexpr (WGT) {
        if (lane < nb) {
          uint64_t o = off[0];
#pragma unroll
          for (int u = 1; u < U; ++u)
            if (lane == u) o = off[u];
          const uint32_t i = (uint32_t)__double2uint_rn((double)o * inv_row_bytes);
          asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(my_wgt + (uint32_t)(stage * U + lane) * 8),
                       "l"(weight + i)
                       : "memory");
        }
      }
      fifo |= (uint32_t)(nb | (pnew ? 0x80 : 0)) << (8 * fifo_pos);
      pnew = false;
      pp += nb;
    }
    asm volatile("cp.async.commit_group;" ::: "memory");  // possibly empty: keeps the group count uniform
  };
#pragma unroll
  for (int s = 0; s < STAGES - 1; ++s) issue(s, s);

  double* __restrict__ Sk = part;
  double acc[VPL][4];
  double run_k = 0.0, run_d = 0.0, run_n = 0.0;  // sums of the rows this lane evaluates (row slot row_of_lane)
  int seg = ~lo;  // < 0: nothing accumulated yet, the first segment is ~seg
  auto load_w = [&](int sgm) {
    seg = sgm;
#pragma unroll
    for (int v = 0; v < VPL; ++v) {
      const int c = col0 + v * 128;
      if (act[v]) {
        const double2 a = *reinterpret_cast<const double2*>(W + (int64_t)seg * D + c);
        const double2 b = *reinterpret_cast<const double2*>(W + (int64_t)seg * D + c + 2);
        asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(my_smem + W_OFF + v * 1024), "d"(a.x), "d"(a.y) : "memory");
        asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(my_smem + W_OFF + v * 1024 + 512), "d"(b.x), "d"(b.y) : "memory");
      }
      acc[v][0] = acc[v][1] = acc[v][2] = acc[v][3] = 0.0;
    }
    run_k = 0.0;
    run_d = 0.0;
    run_n = 0.0;
  };
  auto flush = [&]() {
    // a segment begun by an earlier team: this team's partial goes to cont[team] and acc_cont_kernel adds the
    // partials of all continuing teams, in team order, to the one the segment's first team stored (recomputed here,
    // once per segment, rather than kept live through the row loop)
    const int64_t t_id = (int64_t)blockIdx.x * TEAMS + (threadIdx.x >> 5) / WPR;
    const bool to_cont = offsets[seg] < (int32_t)((int64_t)offsets[M] * t_id / ((int64_t)gridDim.x * TEAMS));
    double* cdst = cont + t_id * (D + CW);
#pragma unroll
    for (int v = 0; v < VPL; ++v) {
      const int c = col0 + v * 128;
      if (act[v]) {
        double* dst = to_cont ? cdst + c : Sk + (int64_t)seg * D + c;
        dst[0] = acc[v][0];  // the only writer of these entries (part is zeroed before the launch)
        dst[1] = acc[v][1];
        dst[2] = acc[v][2];
        dst[3] = acc[v][3];
      }
    }
    // every row slot is evaluated by 32 / U lanes with identical results: count each slot once
    const bool slot_leader = (lane % (32 / U)) == 0;
    const double tk = warp_sum(slot_leader ? run_k : 0.0);
    const double td = warp_sum(slot_leader ? run_d : 0.0);
    const double tn = WGT ? warp_sum(slot_leader ? run_n : 0.0) : 0.0;
    if (tw == 0 && lane == 0) {
      if (to_cont) {
        cdst[D] = tk;
        cdst[D + 1] = td;
        if (WGT) cdst[D + 2] = tn;
        cont_seg[t_id] = seg;
      } else {
        part[(int64_t)M * D + seg] = tk;                      // sk
        part[(int64_t)M * D + 2 * (int64_t)M + seg] = td;     // E
        if (WGT) part[(int64_t)M * D + M + seg] = tn;         // n (the scan wrote the count)
      }
    }
  };

  int stage = 0, parity = 0;
  while (fifo & 0x7fu) {  // batches in flight
    const int nb = (int)(fifo & 0x7fu);
    if (fifo & 0x80u) {  // first batch of a segment: move on to the next segment that has samples
      int nseg = ~seg;
      if (seg >= 0) {
        flush();
        nseg = seg + 1;
        while (offsets[nseg + 1] == offsets[nseg]) ++nseg;
      }
      load_w(nseg);
    }
    fifo >>= 8;
    issue(stage == 0 ? STAGES - 1 : stage - 1, STAGES - 2);  // refill the slot consumed in the previous iteration
    asm volatile("cp.async.wait_group %0;" ::"n"(STAGES - 1) : "memory");
    if constexpr (WGT) __syncwarp();  // the weights are read by the lanes of their row slot, not by the copying lane
    const uint32_t rows = my_smem + (uint32_t)stage * SLOT_BYTES;

    // ALL: the batch has all U rows (the common case) -> no per-row predicates in the unrolled code
    auto body = [&](auto all_tag) {
      constexpr bool ALL = decltype(all_tag)::value;
      double xd[U][VPL][4];
      double part_d2[U];
#pragma unroll
      for (int u = 0; u < U; ++u) part_d2[u] = 0.0;
#pragma unroll
      for (int v = 0; v < VPL; ++v) {
        if (FULLD || act[v]) {
#pragma unroll
          for (int u = 0; u < U; ++u) {
            if (ALL || u < nb) {
              float4 x;
              asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                           : "=f"(x.x), "=f"(x.y), "=f"(x.z), "=f"(x.w)
                           : "r"(rows + (u * VPL + v) * 512));
              // XU of the four conversions go through the XU pipe (F2F.F64.F32, otherwise idle), the rest through the
              // ALU / FMA pipes (four integer instructions each)
              xd[u][v][0] = (double)x.x;
              xd[u][v][1] = XU >= 3 ? (double)x.y : f32_as_f64(x.y);
              xd[u][v][2] = XU >= 2 ? (double)x.z : f32_as_f64(x.z);
              xd[u][v][3] = XU >= 4 ? (double)x.w : f32_as_f64(x.w);
            }
          }
          // the prototype's columns are read once per batch and used for all its rows
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            double w0, w1;
            asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(w0), "=d"(w1) : "r"(my_smem + W_OFF + v * 1024 + h * 512));
#pragma unroll
            for (int u = 0; u < U; ++u) {
              if (ALL || u < nb) {
                const double a = xd[u][v][2 * h] - w0;
                part_d2[u] = fma(a, a, part_d2[u]);
                const double b = xd[u][v][2 * h + 1] - w1;
                part_d2[u] = fma(b, b, part_d2[u]);
              }
            }
          }
        }
      }
      double my_d2 = reduce_rows<U>(part_d2, lane);  // lane l: squared distance of row row_of_lane(l)
      if (WPR > 1) {
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (lane == lane_of_row<U>(u)) red[team][parity][tw][u] = my_d2;
        asm volatile("bar.sync %0, %1;" ::"r"(team + 1), "r"(WPR * 32));
        my_d2 = 0.0;
#pragma unroll
        for (int q = 0; q < WPR; ++q) my_d2 += red[team][parity][q][row_of_lane<U>(lane)];
        parity ^= 1;
      }
      // each lane evaluates the weight and the distance of its row slot (32 / U lanes per slot, redundantly)
      // dbgsom/BaseSom.py:536 squares the distance again; d2 itself is that square to one rounding, and the
      // exponential no longer waits for the square root
      double my_dist = sqrt(my_d2);
      double my_k = 1.0 - sqrt(1.0 - exp(-inv_var * my_d2));
      if constexpr (WGT) {
        double w = 0.0;
        if (ALL || row_of_lane<U>(lane) < nb)
          asm volatile("ld.shared.f64 %0, [%1];" : "=d"(w) : "r"(my_wgt + (uint32_t)(stage * U + row_of_lane<U>(lane)) * 8));
        my_k *= w;  // the k * x sums below take the weighted k
        my_dist *= w;
        run_n += w;
      }
      if (ALL || row_of_lane<U>(lane) < nb) {
        run_k += my_k;
        run_d += my_dist;
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const double k = __shfl_sync(kFullMask, my_k, lane_of_row<U>(u));
        if (ALL || u < nb) {
#pragma unroll
          for (int v = 0; v < VPL; ++v) {
            if (FULLD || act[v]) {
#pragma unroll
              for (int q = 0; q < 4; ++q) acc[v][q] = fma(k, xd[u][v][q], acc[v][q]);
            }
          }
        }
      }
    };
    if (nb == U)
      body(std::true_type{});
    else
      body(std::false_type{});
    if (++stage == STAGES) stage = 0;
  }
  if (seg >= 0) flush();
}

// part[seg] += the partials of the teams that continued segment seg, summed in team order; one CTA per segment (the
// CTA of its first continuing team).  cont_seg is -1 for a team that continued nothing, which includes teams with an
// empty range (fewer samples than teams): those may sit between two teams that continue the same segment and must not
// split its run.  Segments only grow with the team index, so skipping -1 entries never joins two different segments.
// A partial is [Sk (D) | sk | E] or, weighted, [Sk | sk | E | n]: cw = D + 2 or D + 3 entries.
__global__ void __launch_bounds__(256) acc_cont_kernel(const double* __restrict__ cont, const int32_t* __restrict__ cont_seg,
                                                      int64_t n_teams, int M, int D, int cw, double* __restrict__ part) {
  const int64_t t = blockIdx.x;
  const int seg = cont_seg[t];
  if (seg < 0) return;
  for (int64_t u = t - 1; u >= 0; --u) {
    const int q = cont_seg[u];
    if (q == seg) return;  // an earlier team continues seg: its CTA sums the run
    if (q >= 0) break;
  }
  for (int c = threadIdx.x; c < cw; c += blockDim.x) {
    double sum = 0.0;
    for (int64_t u = t; u < n_teams; ++u) {
      const int q = cont_seg[u];
      if (q == seg) sum += cont[u * cw + c];
      else if (q >= 0) break;
    }
    double* dst = c < D ? part + (int64_t)seg * D + c
                        : part + (int64_t)M * D + (c == D ? 0 : c == D + 1 ? 2 * (int64_t)M : (int64_t)M) + seg;
    *dst += sum;
  }
}

constexpr int64_t ACC_MAX_TEAMS = 148 * 2 * 8;  // CTAs (<= 2 per SM) x teams per CTA (<= 8)

template <int VPL, int WPR, int U, int XU, bool WGT>
int launch_accumulate_t(const dbgsom_accumulate_args& a, const double* weight, const int32_t* perm,
                        const int32_t* offsets, double* cont, int32_t* cont_seg, cudaStream_t s) {
  // one warp per row (WPR = 1): 6 warps per CTA leave 168 registers per thread at two CTAs per SM, enough
  // for the U * VPL * 4 converted elements + prototype + sums without spilling (at 128 registers the
  // loop-carried cursors spilled and every iteration stalled on local-memory loads); teams need 8 warps
  constexpr int THREADS = WPR == 1 ? 192 : 256;
  constexpr int STAGES = WPR == 1 ? 4 : 3;
  constexpr int TEAMS = THREADS / 32 / WPR;
  const size_t smem =
      (size_t)(THREADS / 32) * (STAGES * U * VPL * 512 + VPL * 1024 + ACC_WIN_BYTES + (WGT ? STAGES * U * 8 : 0));
  auto kern = a.D == 128 * VPL * WPR ? accumulate_kernel<VPL, WPR, U, THREADS, STAGES, true, XU, WGT>
                                     : accumulate_kernel<VPL, WPR, U, THREADS, STAGES, false, XU, WGT>;
  DBGSOM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 1;  // resident CTAs per SM: 2 by registers (__launch_bounds__) if the staging rings fit twice
  DBGSOM_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, THREADS, smem));
  if (per_sm > 2) per_sm = 2;
  if (per_sm < 1) per_sm = 1;
  int64_t blocks = 148 * per_sm;
  const int64_t useful = ceil_div<int64_t>(ceil_div<int64_t>(a.N, 4 * U), TEAMS);  // >= 4 batches per team
  if (blocks > useful) blocks = useful;
  if (blocks < 1) blocks = 1;
  const int64_t n_teams = blocks * TEAMS;
  static_assert(TEAMS <= 8, "ACC_MAX_TEAMS");
  DBGSOM_CUDA_TRY(cudaMemsetAsync(cont_seg, 0xff, (size_t)n_teams * 4, s));
  kern<<<(unsigned)blocks, THREADS, smem, s>>>(a.d_X, a.N, a.D, a.ldx, perm, offsets, a.d_W, a.M,
                                              a.inv_total_variance, weight, a.d_part, cont, cont_seg);
  DBGSOM_LAUNCH_CHECK();
  acc_cont_kernel<<<(unsigned)n_teams, 256, 0, s>>>(cont, cont_seg, n_teams, a.M, a.D, a.D + (WGT ? 3 : 2), a.d_part);
  DBGSOM_LAUNCH_CHECK();
  return DBGSOM_OK;
}

// the weighted kernels exist for the default variant of each width only (the DBGSOM_ACC_* tuning switches select
// among unweighted variants)
template <int VPL, int WPR, int U, int XU = 1>
int launch_accumulate(const dbgsom_accumulate_args& a, const double* weight, const int32_t* perm, const int32_t* offsets,
                      double* cont, int32_t* cont_seg, cudaStream_t s) {
  if (weight) return DBGSOM_E_UNSUPPORTED;
  return launch_accumulate_t<VPL, WPR, U, XU, false>(a, nullptr, perm, offsets, cont, cont_seg, s);
}
template <int VPL, int WPR, int U, int XU = 1>
int launch_accumulate_w(const dbgsom_accumulate_args& a, const double* weight, const int32_t* perm,
                        const int32_t* offsets, double* cont, int32_t* cont_seg, cudaStream_t s) {
  if (weight) return launch_accumulate_t<VPL, WPR, U, XU, true>(a, weight, perm, offsets, cont, cont_seg, s);
  return launch_accumulate_t<VPL, WPR, U, XU, false>(a, nullptr, perm, offsets, cont, cont_seg, s);
}

// Weighted class histogram per winner, out[j, c] = sum of weight[i] (1 if weight == NULL) over the samples i of
// segment j with label c (float64 [M, n_classes], every cell written).  One warp per segment: lane l adds the weights of positions
// offsets[j] + l, + 32, ... into its own row of shared-memory bins, then the 32 rows are added in lane order -- with
// the stable permutation the sums are the same on every run.  Classes are taken CC at a time.
constexpr int CH_WARPS = 4;
constexpr int CH_CLASSES = 48;
__global__ void __launch_bounds__(CH_WARPS * 32) seg_class_hist_kernel(
    const int32_t* __restrict__ perm, const int32_t* __restrict__ offsets, const int32_t* __restrict__ labels,
    const double* __restrict__ weight, int M, int n_classes, int c0, int cc, double* __restrict__ out) {
  extern __shared__ double ch_bins[];  // [CH_WARPS][32][cc]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j = blockIdx.x * CH_WARPS + warp;
  if (j >= M) return;
  double* bins = ch_bins + (size_t)warp * 32 * cc;
  for (int q = lane; q < 32 * cc; q += 32) bins[q] = 0.0;
  __syncwarp();
  double* mine = bins + lane * cc;
  for (int32_t p = offsets[j] + lane; p < offsets[j + 1]; p += 32) {
    const int32_t i = perm[p];
    const int y = labels[i] - c0;
    if ((unsigned)y < (unsigned)cc) mine[y] += weight ? weight[i] : 1.0;
  }
  __syncwarp();
  for (int c = lane; c < cc; c += 32) {
    double t = 0.0;
    for (int l = 0; l < 32; ++l) t += bins[l * cc + c];
    out[(int64_t)j * n_classes + c0 + c] = t;
  }
}

}  // namespace

struct AccWorkspace {
  int32_t *counts, *offsets, *cursor, *perm;
  int32_t* chunk_table;  // stable scatter: [chunks, M] (dead once perm is built; shares its space with cont)
  double* cont;          // [ACC_MAX_TEAMS, D + 2 (+1 weighted)] partials of teams that continue a segment
  int32_t* cont_seg;     // [ACC_MAX_TEAMS]
  static size_t shared_bytes(int64_t N, int M, int D) {
    const size_t table = M <= STABLE_MAX_M ? (size_t)stable_max_chunks(N) * M * 4 : 0;
    const size_t c = round_up<size_t>((size_t)ACC_MAX_TEAMS * (D + 3) * 8, 256) + (size_t)ACC_MAX_TEAMS * 4;
    return round_up<size_t>(table > c ? table : c, 256);
  }
  static size_t bytes(int64_t N, int M, int D) {
    return 3 * round_up<size_t>((size_t)(M + 1) * 4, 256) + round_up<size_t>((size_t)N * 4, 256) + shared_bytes(N, M, D);
  }
  static AccWorkspace carve(void* base, int64_t N, int M, int D) {
    AccWorkspace w;
    uint8_t* p = reinterpret_cast<uint8_t*>(base);
    const size_t sm = round_up<size_t>((size_t)(M + 1) * 4, 256);
    w.counts = reinterpret_cast<int32_t*>(p);
    w.offsets = reinterpret_cast<int32_t*>(p + sm);
    w.cursor = reinterpret_cast<int32_t*>(p + 2 * sm);
    w.perm = reinterpret_cast<int32_t*>(p + 3 * sm);
    uint8_t* q = p + 3 * sm + round_up<size_t>((size_t)N * 4, 256);
    w.chunk_table = reinterpret_cast<int32_t*>(q);
    w.cont = reinterpret_cast<double*>(q);
    w.cont_seg = reinterpret_cast<int32_t*>(q + round_up<size_t>((size_t)ACC_MAX_TEAMS * (D + 3) * 8, 256));
    return w;
  }
};

size_t accumulate_workspace_bytes(int64_t N, int M, int D) { return AccWorkspace::bytes(N, M, D); }
size_t accumulate_perm_offset(int64_t N, int M) {
  (void)N;
  return 3 * round_up<size_t>((size_t)(M + 1) * 4, 256);
}

// counts per winner (+ the int32 class histogram when class_hist != NULL) -> offsets -> permutation of the samples
// grouped by winner (ascending sample index for M <= STABLE_MAX_M); part_n (may be NULL) receives the counts
static int build_winner_perm(const int32_t* bmu, int64_t N, int M, const int32_t* labels, int n_classes,
                             int32_t* class_hist, const AccWorkspace& ws, double* part_n, cudaStream_t s) {
  DBGSOM_CUDA_TRY(cudaMemsetAsync(ws.counts, 0, (size_t)(M + 1) * 4, s));
  if (class_hist) DBGSOM_CUDA_TRY(cudaMemsetAsync(class_hist, 0, (size_t)M * n_classes * 4, s));
  // histogram
  {
    const int64_t bins = M + (class_hist ? (int64_t)M * n_classes : 0);
    const bool smem = bins <= HIST_SMEM_BINS;
    const int64_t rows_per_block = smem ? 16384 : 4096;
    const unsigned blocks = (unsigned)ceil_div<int64_t>(N, rows_per_block);
    if (smem)
      hist_kernel<true><<<blocks, HIST_THREADS, (size_t)bins * 4, s>>>(bmu, N, M, class_hist ? labels : nullptr,
                                                                     n_classes, ws.counts, class_hist, rows_per_block);
    else
      hist_kernel<false><<<blocks, HIST_THREADS, 0, s>>>(bmu, N, M, class_hist ? labels : nullptr, n_classes, ws.counts,
                                                        class_hist, rows_per_block);
    DBGSOM_LAUNCH_CHECK();
  }
  scan_kernel<<<1, SCAN_THREADS, 0, s>>>(ws.counts, M, ws.offsets, ws.cursor, part_n);
  DBGSOM_LAUNCH_CHECK();
  if (M <= STABLE_MAX_M) {
    const StableChunks sc = stable_chunks(N, M);
    const size_t smem = (size_t)sc.warps * M * 4;
    const unsigned ctas = (unsigned)ceil_div<int64_t>(sc.n, sc.warps);
    DBGSOM_CUDA_TRY(cudaFuncSetAttribute(stable_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    DBGSOM_CUDA_TRY(cudaFuncSetAttribute(stable_place_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    stable_count_kernel<<<ctas, sc.warps * 32, smem, s>>>(bmu, N, M, sc.chunk, sc.n, ws.chunk_table);
    DBGSOM_LAUNCH_CHECK();
    stable_base_kernel<<<(unsigned)ceil_div(M, 32), 1024, 0, s>>>(ws.chunk_table, sc.n, M, ws.offsets);
    DBGSOM_LAUNCH_CHECK();
    stable_place_kernel<<<ctas, sc.warps * 32, smem, s>>>(bmu, N, M, sc.chunk, sc.n, ws.chunk_table, ws.perm);
    DBGSOM_LAUNCH_CHECK();
  } else {  // maps too large for the per-warp tables: slots in arrival order
    int64_t blocks = ceil_div<int64_t>(N, SCAT_THREADS * 4);
    if (blocks > 148 * 16) blocks = 148 * 16;
    scatter_kernel<<<(unsigned)blocks, SCAT_THREADS, 0, s>>>(bmu, N, M, ws.offsets, ws.cursor, ws.perm);
    DBGSOM_LAUNCH_CHECK();
  }
  return DBGSOM_OK;
}

// float64 [M, n_classes] weighted class histogram over the segments of a permutation built by build_winner_perm
static int run_seg_class_hist(const AccWorkspace& ws, const int32_t* labels, const double* weight, int M, int n_classes,
                              double* out, cudaStream_t s) {
  const int cc_max = n_classes < CH_CLASSES ? n_classes : CH_CLASSES;
  DBGSOM_CUDA_TRY(cudaFuncSetAttribute(seg_class_hist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       CH_WARPS * 32 * cc_max * 8));
  for (int c0 = 0; c0 < n_classes; c0 += CH_CLASSES) {
    const int cc = n_classes - c0 < CH_CLASSES ? n_classes - c0 : CH_CLASSES;
    seg_class_hist_kernel<<<(unsigned)ceil_div(M, CH_WARPS), CH_WARPS * 32, (size_t)CH_WARPS * 32 * cc * 8, s>>>(
        ws.perm, ws.offsets, labels, weight, M, n_classes, c0, cc, out);
    DBGSOM_LAUNCH_CHECK();
  }
  return DBGSOM_OK;
}

size_t label_hist_weighted_workspace_bytes(int64_t N, int M) { return AccWorkspace::bytes(N, M, 1); }

int run_label_counts_weighted(const int32_t* idx, const int32_t* labels, const double* weight, int64_t N, int M,
                              int n_classes, double* counts, void* workspace, cudaStream_t s) {
  const AccWorkspace ws = AccWorkspace::carve(workspace, N, M, 1);
  const int rc = build_winner_perm(idx, N, M, nullptr, 0, nullptr, ws, nullptr, s);
  if (rc != DBGSOM_OK) return rc;
  return run_seg_class_hist(ws, labels, weight, M, n_classes, counts, s);
}

int run_accumulate(const dbgsom_accumulate_args& a, const double* weight, double* class_hist_w, cudaStream_t s) {
  const AccWorkspace ws = AccWorkspace::carve(a.d_workspace, a.N, a.M, a.D);
  const int64_t M = a.M, D = a.D;
  DBGSOM_CUDA_TRY(cudaMemsetAsync(a.d_part, 0, (size_t)(M * D + 3 * M) * sizeof(double), s));
  const bool with_labels = a.d_labels != nullptr && a.n_classes > 0 &&
                           (weight ? class_hist_w != nullptr : a.d_class_hist != nullptr);
  // weighted: the class histogram is summed per segment after the scatter (float64, fixed order)
  int rc = build_winner_perm(a.d_bmu, a.N, a.M, a.d_labels, a.n_classes,
                             with_labels && !weight ? a.d_class_hist : nullptr, ws, a.d_part + M * D + M, s);
  if (rc != DBGSOM_OK) return rc;
  if (with_labels && weight) {
    rc = run_seg_class_hist(ws, a.d_labels, weight, a.M, a.n_classes, class_hist_w, s);
    if (rc != DBGSOM_OK) return rc;
  }
  const int D4 = a.D;
  static const char* tune_u = getenv("DBGSOM_ACC_ROWS");  // tuning switch: rows per batch for D <= 256
  const int u_small = tune_u ? atoi(tune_u) : 0;
  // float -> double conversions on the XU pipe (F2F) per float4; the rest take four integer instructions each on the
  // ALU / FMA pipes.  Default: all four -- with the lean loop control the kernel is short of issue slots, not of XU
  // cycles (ncu: XU 20 % busy at two in four).  10M x 256 rows stand-alone 1.80 (one) / 1.76 (two) / 1.72 ms (four);
  // in the bench epoch, at the clock K1 leaves, 2.21 / 2.17 / 2.12 ms.  DBGSOM_ACC_XU=1..4 selects.
  static const char* tune_xu = getenv("DBGSOM_ACC_XU");
  const int xu = weight ? 4 : (tune_xu ? atoi(tune_xu) : 4);
  const double* w = weight;
  if (D4 <= 128) {
    if (u_small == 4 && !w) return launch_accumulate<1, 1, 4>(a, w, ws.perm, ws.offsets, ws.cont, ws.cont_seg, s);
    if (xu >= 4) return launch_accumulate_w<1, 1, 8, 4>(a, w, ws.perm, ws.offsets, ws.cont, ws.cont_seg, s);
    if (xu == 3) return launch_accumulate<1, 1, 8, 3>(a, w, ws.perm, ws.offsets, ws.cont, ws.cont_seg, s);
    if (xu == 2) return launch_accumulate<1, 1, 8, 2>(a, w, ws.perm, ws.offsets, ws.cont, ws.cont_seg, s);
    return launch_accumulate<1, 1, 8>(a, w, ws.perm, ws.offsets, ws.cont, ws.cont_seg, s);
  }
  if (D4 <= 256) {
    if (u_small == 2 && !w) return launch_accumulate<2, 1, 2>(a, w, ws.perm, ws.offsets, ws.cont, ws.cont_seg, s);
    if (xu >= 4) return launch_accumulate_w<2, 1, 4, 4>(a, w, ws.perm, ws.offsets, ws.cont, ws.cont_seg, s);
    if (xu == 3) return launch_accumulate<2, 1, 4, 3>(a, w, ws.perm, ws.offsets, ws.cont, ws.cont_seg, s);
    if (xu == 2) return launch_accumulate<2, 1, 4, 2>(a, w, ws.perm, ws.offsets, ws.cont, ws.cont_seg, s);
    return launch_accumulate<2, 1, 4>(a, w, ws.perm, ws.offsets, ws.cont, ws.cont_seg, s);
  }
  if (D4 <= 512) return launch_accumulate_w<4, 1, 2>(a, w, ws.perm, ws.offsets, ws.cont, ws.cont_seg, s);
  if (D4 <= 1024) return launch_accumulate_w<4, 2, 2>(a, w, ws.perm, ws.offsets, ws.cont, ws.cont_seg, s);
  if (D4 <= 2048) return launch_accumulate_w<4, 4, 2>(a, w, ws.perm, ws.offsets, ws.cont, ws.cont_seg, s);
  if (D4 <= 4096) return launch_accumulate_w<4, 8, 2>(a, w, ws.perm, ws.offsets, ws.cont, ws.cont_seg, s);
  return DBGSOM_E_UNSUPPORTED;
}

}  // namespace dbgsom
