// K3: neighbourhood smoothing  W <- (H . (n * C')) / (H . n)  in float64.
//
// Replaces (dbgsom/BaseSom.py): _calculate_gaussian_neighborhood :525-531 (H = exp(-hop^2/2sigma^2),
// taken here from a host-computed table indexed by the integer hop count, bit-identical to the
// reference's np.exp), Step 4 :509-515 (the reference materialises an M x M x D broadcast; this is
// the same sum as a GEMM) and Step 5 :518-522 (sum_i ||W_i - W_new_i||).
// Centres follow the reference's row packing (quirk Q1) when pack_rows != 0.
#include "common.cuh"

namespace dbgsom {

namespace {

// ------------------------------------------------------------------------------------------ centres
// single CTA: rank live neurons (n > 0), src[r] = index of the r-th live neuron (or -1)
constexpr int RANK_THREADS = 1024;
__global__ void __launch_bounds__(RANK_THREADS) live_rank_kernel(const double* __restrict__ n, int M, int pack,
                                                                int32_t* __restrict__ src, int32_t* __restrict__ live_list,
                                                                double* __restrict__ n_live_vals,
                                                                int32_t* __restrict__ n_live) {
  __shared__ int32_t warp_tot[32];
  __shared__ int32_t carry_sh;
  if (threadIdx.x == 0) carry_sh = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int base = 0; base < M; base += RANK_THREADS) {
    const int j = base + threadIdx.x;
    const int live = (j < M && n[j] > 0.0) ? 1 : 0;
    if (j < M) src[j] = pack ? -1 : (live ? j : -1);
    __syncthreads();  // all -1 defaults of this pass are written before any rank lands (rank <= j)
    int v = live;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(kFullMask, v, o);
      if (lane >= o) v += t;
    }
    if (lane == 31) warp_tot[warp] = v;
    __syncthreads();
    if (warp == 0) {
      int t = warp_tot[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(kFullMask, t, o);
        if (lane >= o) t += u;
      }
      warp_tot[lane] = t;
    }
    __syncthreads();
    const int carry = carry_sh;
    const int rank = carry + (warp ? warp_tot[warp - 1] : 0) + v - live;
    if (pack && live) src[rank] = j;  // rank <= j: never clobbers a default written by a later pass
    if (live) {  // compact list of the neurons that won samples: the only columns of H that matter
      live_list[rank] = j;
      n_live_vals[rank] = n[j];
    }
    __syncthreads();
    if (threadIdx.x == RANK_THREADS - 1) carry_sh = carry + warp_tot[31];
    __syncthreads();
  }
  if (threadIdx.x == 0) *n_live = carry_sh;
}

// Only neurons with samples (n_j > 0) contribute to either sum of the update, so both run over the compact
// list live[0..L):  Bc[r, :] = n_j * C'[j, :],  j = live[r],  C'[j] = Sk[src_j] / sk[src_j]  (0 when src_j < 0:
// with packed rows a live neuron beyond the first L rows has an all-zero centre, quirk Q1).
__global__ void __launch_bounds__(256) weighted_centres_kernel(const double* __restrict__ part, int M, int D,
                                                              const int32_t* __restrict__ src,
                                                              const int32_t* __restrict__ live,
                                                              const int32_t* __restrict__ n_live,
                                                              double* __restrict__ Bc) {
  const double* Sk = part;
  const double* sk = part + (int64_t)M * D;
  const double* n = sk + M;
  const int64_t total = (int64_t)(*n_live) * D;
  for (int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x; e < total; e += (int64_t)gridDim.x * 256) {
    const int r = (int)(e / D), d = (int)(e % D);
    const int j = live[r];
    const int sj = src[j];
    Bc[e] = sj >= 0 ? n[j] * (Sk[(int64_t)sj * D + d] / sk[sj]) : 0.0;
  }
}

// den[i] = sum_r H[i, live[r]] n[live[r]]  for the rows [row_begin, row_end)
__global__ void __launch_bounds__(256) denominator_kernel(const uint16_t* __restrict__ hop, int64_t ldh,
                                                         const double* __restrict__ lut, int lut_len,
                                                         const int32_t* __restrict__ live,
                                                         const double* __restrict__ n_live_vals,
                                                         const int32_t* __restrict__ n_live, int row_begin,
                                                         int row_end, double* __restrict__ den) {
  const int lane = threadIdx.x & 31;
  const int i = row_begin + blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= row_end) return;
  const int L = *n_live;
  double acc = 0.0;
  for (int r = lane; r < L; r += 32) {
    const unsigned h = hop[(int64_t)i * ldh + live[r]];
    if (h < (unsigned)lut_len) acc = fma(lut[h], n_live_vals[r], acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) den[i] = acc;
}

// ------------------------------------------------------------------------------------------ GEMM
// W_out[i, d] = (sum_r H[i, live[r]] Bc[r, d]) / den[i] for rows [row_begin, row_end);   tile 128 (i) x 64 (d),
// 16-wide steps over the live list, 8 x 4 outputs per thread (6 shared-memory vector loads per 32 DFMA keeps
// the float64 pipe, not the LDS port, the limiter).
constexpr int TI = 128, TD = 64, TJ = 16;
__global__ void __launch_bounds__(256, 2) smooth_gemm_kernel(const uint16_t* __restrict__ hop, int64_t ldh,
                                                         const double* __restrict__ lut, int lut_len,
                                                         const double* __restrict__ B, const double* __restrict__ den,
                                                         const int32_t* __restrict__ live,
                                                         const int32_t* __restrict__ n_live, int row_begin,
                                                         int row_end, int D, double* __restrict__ W_out) {
  __shared__ __align__(16) double Hs[TJ][TI];
  __shared__ __align__(16) double Bs[TJ][TD];
  const int tid = threadIdx.x;
  const int tx = tid % 16;  // 4 columns
  const int ty = tid / 16;  // 8 rows
  const int i0 = row_begin + blockIdx.y * TI, d0 = blockIdx.x * TD;
  const int L = *n_live;
  double acc[8][4] = {};

  // Software pipeline: the next step's H entries (hop -> table lookup: two dependent loads) and B entries are fetched
  // into registers while the current step is computed from shared memory; the first version loaded, synchronised,
  // computed and synchronised again, with the global-load latency exposed once per 16 live neurons (~35 % of the
  // float64 pipe).
  const int ii = tid >> 1, jj0 = (tid & 1) * 8;  // H tile: thread -> (i = tid / 2, 8 consecutive j)
  const int hi_row = i0 + ii;
  double hq[8], bq[4];
  auto fetch = [&](int j0) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int j = j0 + jj0 + q;
      double h = 0.0;
      if (hi_row < row_end && j < L) {
        const unsigned hp = hop[(int64_t)hi_row * ldh + live[j]];
        if (hp < (unsigned)lut_len) h = lut[hp];
      }
      hq[q] = h;
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int e = tid + q * 256;
      const int j = j0 + e / TD, d = d0 + e % TD;
      bq[q] = (j < L && d < D) ? B[(int64_t)j * D + d] : 0.0;
    }
  };
  if (L > 0) fetch(0);
  for (int j0 = 0; j0 < L; j0 += TJ) {
#pragma unroll
    for (int q = 0; q < 8; ++q) Hs[jj0 + q][ii] = hq[q];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int e = tid + q * 256;
      Bs[e / TD][e % TD] = bq[q];
    }
    __syncthreads();
    if (j0 + TJ < L) fetch(j0 + TJ);
#pragma unroll
    for (int jj = 0; jj < TJ; ++jj) {
      double h[8];
#pragma unroll
      for (int r = 0; r < 8; r += 2) {
        const double2 hv = *reinterpret_cast<const double2*>(&Hs[jj][ty * 8 + r]);
        h[r] = hv.x;
        h[r + 1] = hv.y;
      }
      const double2 b01 = *reinterpret_cast<const double2*>(&Bs[jj][tx * 4]);
      const double2 b23 = *reinterpret_cast<const double2*>(&Bs[jj][tx * 4 + 2]);
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        acc[r][0] = fma(h[r], b01.x, acc[r][0]);
        acc[r][1] = fma(h[r], b01.y, acc[r][1]);
        acc[r][2] = fma(h[r], b23.x, acc[r][2]);
        acc[r][3] = fma(h[r], b23.y, acc[r][3]);
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int i = i0 + ty * 8 + r;
    if (i >= row_end) continue;
    const double dn = den[i];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int d = d0 + tx * 4 + c;
      if (d < D) W_out[(int64_t)i * D + d] = acc[r][c] / dn;
    }
  }
}

// row_norm[i] = ||W_in[i] - W_out[i]||_2, one warp per row
__global__ void __launch_bounds__(256) change_kernel(const double* __restrict__ W_in, const double* __restrict__ W_out,
                                                    int row_begin, int row_end, int D, double* __restrict__ row_norm) {
  const int lane = threadIdx.x & 31;
  const int i = row_begin + blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= row_end) return;
  double acc = 0.0;
  for (int d = lane; d < D; d += 32) {
    const double t = W_in[(int64_t)i * D + d] - W_out[(int64_t)i * D + d];
    acc = fma(t, t, acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) row_norm[i] = sqrt(acc);
}

// change += sum of row_norm[row_begin:row_end], one CTA, in a fixed order (the same value on every run)
constexpr int CHANGE_SUM_THREADS = 1024;
__global__ void __launch_bounds__(CHANGE_SUM_THREADS) change_sum_kernel(const double* __restrict__ row_norm,
                                                                       int row_begin, int row_end,
                                                                       double* __restrict__ change) {
  __shared__ double part[CHANGE_SUM_THREADS / 32];
  double acc = 0.0;
  for (int i = row_begin + threadIdx.x; i < row_end; i += CHANGE_SUM_THREADS) acc += row_norm[i];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double total = 0.0;
    for (int w = 0; w < CHANGE_SUM_THREADS / 32; ++w) total += part[w];
    *change += total;
  }
}

}  // namespace

struct SmoothWorkspace {
  int32_t *src, *live, *n_live;
  double *den, *n_live_vals, *B;
  static size_t bytes(int M, int D) {
    return 2 * round_up<size_t>((size_t)M * 4, 256) + 256 + 2 * round_up<size_t>((size_t)M * 8, 256) + (size_t)M * D * 8;
  }
  static SmoothWorkspace carve(void* base, int M, int D) {
    SmoothWorkspace w;
    uint8_t* p = reinterpret_cast<uint8_t*>(base);
    w.src = reinterpret_cast<int32_t*>(p);
    p += round_up<size_t>((size_t)M * 4, 256);
    w.live = reinterpret_cast<int32_t*>(p);
    p += round_up<size_t>((size_t)M * 4, 256);
    w.n_live = reinterpret_cast<int32_t*>(p);
    p += 256;
    w.den = reinterpret_cast<double*>(p);
    p += round_up<size_t>((size_t)M * 8, 256);
    w.n_live_vals = reinterpret_cast<double*>(p);
    p += round_up<size_t>((size_t)M * 8, 256);
    w.B = reinterpret_cast<double*>(p);
    return w;
  }
};

size_t smooth_workspace_bytes(int M, int D) { return SmoothWorkspace::bytes(M, D); }

int run_smooth(const dbgsom_smooth_args& a, cudaStream_t s) {
  const SmoothWorkspace ws = SmoothWorkspace::carve(a.d_workspace, a.M, a.D);
  const int M = a.M, D = a.D;
  const int r0 = a.row_end > a.row_begin ? a.row_begin : 0;
  const int r1 = a.row_end > a.row_begin ? a.row_end : M;
  const int rows = r1 - r0;
  const double* n = a.d_part + (int64_t)M * D + M;
  DBGSOM_CUDA_TRY(cudaMemsetAsync(a.d_change, 0, sizeof(double), s));
  live_rank_kernel<<<1, RANK_THREADS, 0, s>>>(n, M, a.pack_rows, ws.src, ws.live, ws.n_live_vals, ws.n_live);
  DBGSOM_LAUNCH_CHECK();
  {
    int64_t blocks = ceil_div<int64_t>((int64_t)M * D, 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    weighted_centres_kernel<<<(unsigned)blocks, 256, 0, s>>>(a.d_part, M, D, ws.src, ws.live, ws.n_live, ws.B);
    DBGSOM_LAUNCH_CHECK();
  }
  denominator_kernel<<<ceil_div(rows, 8), 256, 0, s>>>(a.d_hop, a.ldh, a.d_kernel_lut, a.lut_len, ws.live,
                                                       ws.n_live_vals, ws.n_live, r0, r1, ws.den);
  DBGSOM_LAUNCH_CHECK();
  {
    const dim3 grid(ceil_div(D, TD), ceil_div(rows, TI));
    smooth_gemm_kernel<<<grid, 256, 0, s>>>(a.d_hop, a.ldh, a.d_kernel_lut, a.lut_len, ws.B, ws.den, ws.live, ws.n_live,
                                            r0, r1, D, a.d_W_out);
    DBGSOM_LAUNCH_CHECK();
  }
  // the row norms go to ws.B (the GEMM above was its last reader)
  change_kernel<<<ceil_div(rows, 8), 256, 0, s>>>(a.d_W_in, a.d_W_out, r0, r1, D, ws.B);
  DBGSOM_LAUNCH_CHECK();
  change_sum_kernel<<<1, CHANGE_SUM_THREADS, 0, s>>>(ws.B, r0, r1, a.d_change);
  DBGSOM_LAUNCH_CHECK();
  return DBGSOM_OK;
}

}  // namespace dbgsom
