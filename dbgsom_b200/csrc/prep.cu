// K4 column statistics, fp16 shadows, and the small prototype-row utilities.
#include "common.cuh"

namespace dbgsom {

namespace {

// ------------------------------------------------------------------------------------------ K4
// Part r = blockIdx.y of moments ([DBGSOM_COLSTATS_PARTS][2D + 1]) gets the rows of row block r:
// [d] = sum_i (x_id - c_d), [D + d] = sum_i (x_id - c_d)^2 (float64), [2D] = max |x_id - c_d| over its columns.
// No atomics: the caller adds the parts in order, so the statistics are the same on every run.
// Replaces np.var(data, axis=0) / np.std(data, axis=0, ddof=1), dbgsom/BaseSom.py:363, :380.
// Shifting by a data row keeps the one-pass variance free of cancellation.
// WGT: the moments are weighted, w_i (x_id - c_d) and w_i (x_id - c_d)^2; the maximum stays over every row (all rows,
// zero-weight ones included, go through the fp16 shadow that it scales).
constexpr int CS_COLS = 32, CS_ROWS = 8;
template <bool WGT>
__global__ void __launch_bounds__(CS_COLS * CS_ROWS) colstats_kernel(const float* __restrict__ X, int64_t N, int D,
                                                                    int64_t ldx, const float* __restrict__ shift,
                                                                    const double* __restrict__ weight,
                                                                    double* __restrict__ moments,
                                                                    int64_t rows_per_block) {
  __shared__ double s1[CS_ROWS][CS_COLS], s2[CS_ROWS][CS_COLS], s3[CS_ROWS][CS_COLS];
  const int cx = threadIdx.x % CS_COLS, ry = threadIdx.x / CS_COLS;
  const int d = blockIdx.x * CS_COLS + cx;
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_block;
  const int64_t r1 = r0 + rows_per_block < N ? r0 + rows_per_block : N;
  double a1 = 0.0, a2 = 0.0, a3 = 0.0;
  if (d < D) {
    const float c = shift[d];
    for (int64_t r = r0 + ry; r < r1; r += CS_ROWS) {
      const double t = (double)X[r * ldx + d] - (double)c;
      const double wt = WGT ? weight[r] * t : t;
      a1 += wt;
      a2 = fma(wt, t, a2);
      a3 = fmax(a3, fabs(t));
    }
  }
  s1[ry][cx] = a1;
  s2[ry][cx] = a2;
  s3[ry][cx] = a3;
  __syncthreads();
  if (ry == 0 && d < D) {
#pragma unroll
    for (int q = 1; q < CS_ROWS; ++q) {
      a1 += s1[q][cx];
      a2 += s2[q][cx];
      a3 = fmax(a3, s3[q][cx]);
    }
    double* part = moments + (int64_t)blockIdx.y * (2 * D + 1);
    part[d] = a1;
    part[D + d] = a2;
    // non-negative doubles order like their bit patterns (the column blocks of a part share this entry)
    atomicMax(reinterpret_cast<long long*>(&part[2 * D]), __double_as_longlong(a3));
  }
}

// ------------------------------------------------------------------------------------------ shadows
// x' = (X[i, :] - shift) * scale;  X16_hi = half(x'), X16_lo = half(x' - X16_hi) (optional), zero
// padded to ld16;  xnorm16[i] = ||x'||_2 rounded up.  With `perm`, shadow row p is built from sample perm[p]
// (sorted sample order of the selective search); xnorm16 stays indexed by sample.
__global__ void __launch_bounds__(256) prepare_x16_kernel(const float* __restrict__ X, int64_t N, int D, int64_t ldx,
                                                         const float* __restrict__ shift, float scale,
                                                         const int32_t* __restrict__ perm,
                                                         __half* __restrict__ X16_hi, __half* __restrict__ X16_lo,
                                                         int64_t ld16, float* __restrict__ xnorm16) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= N) return;
  const int64_t src = perm ? (int64_t)perm[row] : row;
  float acc = 0.f;
  for (int64_t d = lane * 2; d < ld16; d += 64) {
    float v0 = 0.f, v1 = 0.f;
    if (d < D) v0 = (X[src * ldx + d] - shift[d]) * scale;
    if (d + 1 < D) v1 = (X[src * ldx + d + 1] - shift[d + 1]) * scale;
    v0 = fminf(fmaxf(v0, -65504.f), 65504.f);  // the host picks `scale` so that this never binds
    v1 = fminf(fmaxf(v1, -65504.f), 65504.f);
    const __half2 h = __floats2half2_rn(v0, v1);
    *reinterpret_cast<__half2*>(X16_hi + row * ld16 + d) = h;
    if (X16_lo) {
      const float2 f = __half22float2(h);
      *reinterpret_cast<__half2*>(X16_lo + row * ld16 + d) = __floats2half2_rn(v0 - f.x, v1 - f.y);
    }
    acc = fmaf(v0, v0, acc);
    acc = fmaf(v1, v1, acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) xnorm16[src] = sqrtf(acc) * (1.f + 1e-6f);
}

// column means of W (float64): wshift[d] = mean_j W[j, d]
__global__ void __launch_bounds__(256) w_colmean_kernel(const double* __restrict__ W, int M, int D,
                                                       double* __restrict__ wshift) {
  const int d = blockIdx.x * 32 + (threadIdx.x & 31);
  const int ry = threadIdx.x >> 5;
  __shared__ double part[8][32];
  double acc = 0.0;
  if (d < D)
    for (int j = ry; j < M; j += 8) acc += W[(int64_t)j * D + d];
  part[ry][threadIdx.x & 31] = acc;
  __syncthreads();
  if (ry == 0 && d < D) {
#pragma unroll
    for (int q = 1; q < 8; ++q) acc += part[q][threadIdx.x & 31];
    wshift[d] = acc / (double)M;
  }
}

// W32 = float(W).  With u = (W - wshift) * scale and v = (wshift - shift) * scale:
// W16_hi = half(u), W16_lo = half(u - W16_hi) (zero rows up to Mpad), wnorm = ||u||^2 + 2 u.v
// wmax = { max ||u_j||_2, max ||w_j||_2, max |wnorm_j|, max |u_jd| } (float bits, atomicMax as int; all >= 0)
__global__ void __launch_bounds__(128) prepare_w_kernel(const double* __restrict__ W, int M, int D,
                                                       const float* __restrict__ shift,
                                                       const double* __restrict__ wshift, float scale,
                                                       float* __restrict__ W32, __half* __restrict__ W16_hi,
                                                       __half* __restrict__ W16_lo, int64_t ld16,
                                                       const int32_t* __restrict__ col_of_proto,
                                                       float* __restrict__ wnorm, float* __restrict__ wmax) {
  __shared__ double red[3][4];
  const int j = blockIdx.x;
  const int64_t col = col_of_proto ? col_of_proto[j] : j;  // shadow position of prototype (or padding) j
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double nu = 0.0, nr = 0.0, uv = 0.0;
  float uinf = 0.f;
  const __half zero = __float2half_rn(0.f);
  if (j < M) {
    for (int d = threadIdx.x; d < D; d += 128) {
      const double w = W[(int64_t)j * D + d];
      W32[(int64_t)j * D + d] = (float)w;
      nr = fma(w, w, nr);
      if (W16_hi) {
        const double c = wshift[d];
        const double u = (w - c) * (double)scale;
        const double v = (c - (double)shift[d]) * (double)scale;
        nu = fma(u, u, nu);
        uv = fma(u, v, uv);
        uinf = fmaxf(uinf, fabsf((float)u));
        const __half h = __float2half_rn(fminf(fmaxf((float)u, -65504.f), 65504.f));
        W16_hi[col * ld16 + d] = h;
        if (W16_lo) W16_lo[col * ld16 + d] = __float2half_rn((float)(u - (double)__half2float(h)));
      }
    }
    if (W16_hi)
      for (int64_t d = D + threadIdx.x; d < ld16; d += 128) {
        W16_hi[col * ld16 + d] = zero;
        if (W16_lo) W16_lo[col * ld16 + d] = zero;
      }
  } else if (W16_hi) {
    for (int64_t d = threadIdx.x; d < ld16; d += 128) {
      W16_hi[col * ld16 + d] = zero;
      if (W16_lo) W16_lo[col * ld16 + d] = zero;
    }
  }
  nu = warp_sum(nu);
  nr = warp_sum(nr);
  uv = warp_sum(uv);
  uinf = warp_max(uinf);
  // |u| beyond the fp16 range is clamped above; the host sees it in wmax[3] and redoes the epoch in fp32
  if (lane == 0 && uinf > 0.f) atomicMax(reinterpret_cast<int*>(wmax + 3), __float_as_int(uinf));
  if (lane == 0) {
    red[0][warp] = nu;
    red[1][warp] = nr;
    red[2][warp] = uv;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    nu = red[0][0] + red[0][1] + red[0][2] + red[0][3];
    nr = red[1][0] + red[1][1] + red[1][2] + red[1][3];
    uv = red[2][0] + red[2][1] + red[2][2] + red[2][3];
    const double bias = nu + 2.0 * uv;
    if (wnorm) wnorm[col] = j < M ? (float)bias : __int_as_float(0x7f800000);
    if (j < M) {
      // round up so the stored maxima are upper bounds
      atomicMax(reinterpret_cast<int*>(wmax + 0), __float_as_int(__double2float_ru(sqrt(nu))));
      atomicMax(reinterpret_cast<int*>(wmax + 1), __float_as_int(__double2float_ru(sqrt(nr))));
      atomicMax(reinterpret_cast<int*>(wmax + 2), __float_as_int(__double2float_ru(fabs(bias))));
    }
  }
}

// ------------------------------------------------------------------------------------------ tile bounds
// Per 128 shadow columns: max ||u_j|| and max |wnorm_j| over the prototypes stored there (padding columns and
// prototypes taken out of the search -- wnorm = +inf -- do not count).  One CTA per tile, a warp per column; the
// maxima are rounded up so that they stay upper bounds.  Feeds the per-tile error bounds of the candidate search
// (bmu_tc.cu, TB).
__global__ void __launch_bounds__(256) tile_bounds_kernel(const double* __restrict__ W, int M, int D,
                                                         const double* __restrict__ wshift, float scale,
                                                         const int32_t* __restrict__ proto_of_col,
                                                         const float* __restrict__ wnorm, float* __restrict__ out) {
  __shared__ float red[2][8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float um = 0.f, wm = 0.f;
  for (int i = warp; i < 128; i += 8) {
    const int c = blockIdx.x * 128 + i;
    const int j = proto_of_col ? proto_of_col[c] : c;
    const float wn = wnorm[c];
    if (j < 0 || j >= M || !(fabsf(wn) < 3.0e38f)) continue;  // warp-uniform
    double nu = 0.0;
    for (int d = lane; d < D; d += 32) {
      const double u = (W[(int64_t)j * D + d] - wshift[d]) * (double)scale;
      nu = fma(u, u, nu);
    }
    nu = warp_sum(nu);
    um = fmaxf(um, __double2float_ru(sqrt(nu)));
    wm = fmaxf(wm, fabsf(wn));
  }
  if (lane == 0) {
    red[0][warp] = um;
    red[1][warp] = wm;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int q = 1; q < 8; ++q) {
      um = fmaxf(um, red[0][q]);
      wm = fmaxf(wm, red[1][q]);
    }
    out[2 * blockIdx.x] = um;
    out[2 * blockIdx.x + 1] = wm;
  }
}

// ------------------------------------------------------------------------------------------ duplicates
// Exact copies among the prototypes.  The reference breaks exact distance ties by the lowest index
// (sklearn/utils/_heap.pyx:46), so a prototype that equals a LOWER-indexed one element by element can never be
// the answer of a top-1 search: its wnorm is set to +inf, which takes it out of the tensor candidate search.
// With the copies gone, equal approximate scores no longer need to be ordered by prototype index in the
// epilogue (bmu_tc.cu, args.ties_any) -- on collapsed maps that ordering was most of its work.
// Step 1: an order-independent 64-bit hash of every row (values, so that -0.0 == +0.0 hash alike).
__device__ __forceinline__ uint64_t mix64(uint64_t z) {  // splitmix64 finaliser
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}
__global__ void __launch_bounds__(128) row_hash_kernel(const double* __restrict__ W, int M, int D,
                                                      unsigned long long* __restrict__ hash) {
  __shared__ unsigned long long part[4];
  const int j = blockIdx.x;
  unsigned long long h = 0;
  for (int d = threadIdx.x; d < D; d += 128) {
    const double w = W[(int64_t)j * D + d] + 0.0;  // -0.0 -> +0.0
    h += mix64((uint64_t)__double_as_longlong(w) + 0x9e3779b97f4a7c15ull * (uint64_t)(d + 1));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) h += __shfl_xor_sync(kFullMask, h, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = h;
  __syncthreads();
  if (threadIdx.x == 0) hash[j] = part[0] + part[1] + part[2] + part[3];
}
// Step 2: one thread per prototype j looks for an equal hash among the lower indices -- tiles of 256 hashes
// staged in shared memory, compared branch-free -- and confirms a hit element by element (lowest index first).
__global__ void __launch_bounds__(256) mark_duplicates_kernel(const double* __restrict__ W, int M, int D,
                                                             const unsigned long long* __restrict__ hash,
                                                             const int32_t* __restrict__ col_of_proto,
                                                             float* __restrict__ wnorm) {
  __shared__ unsigned long long tile[256];
  const int j = blockIdx.x * 256 + threadIdx.x;
  const unsigned long long hj = j < M ? hash[j] : 0ull;
  bool done = j >= M;
  for (int t = 0; t <= (int)blockIdx.x; ++t) {  // block-uniform trip count
    __syncthreads();
    const int src = t * 256 + threadIdx.x;
    tile[threadIdx.x] = src < M ? hash[src] : 0ull;
    __syncthreads();
    if (done) continue;
    const int lim = min(256, j - t * 256);  // only lower indices
    bool hit = false;
#pragma unroll 16
    for (int q = 0; q < 256; ++q) hit |= (tile[q] == hj) & (q < lim);
    if (!hit) continue;
    for (int q = 0; q < lim && !done; ++q) {
      if (tile[q] != hj) continue;
      const int p = t * 256 + q;
      bool same = true;
      for (int d = 0; d < D && same; ++d) same = W[(int64_t)p * D + d] == W[(int64_t)j * D + d];
      if (same) {
        wnorm[col_of_proto ? col_of_proto[j] : j] = __int_as_float(0x7f800000);
        done = true;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------ bias rows
// wnorm folded into the MMA: the candidate kernel ends every output tile with one extra k-step whose A operand is
// the constant E = 2^e in its first three columns and whose B operand holds three fp16 pieces (h, m, l) of
// -wnorm_j / (2 E) in the first three columns of Wb16[c, :] (c = shadow row), so the accumulator becomes
// x'.u - wnorm/2 = -score/2 and the epilogue needs no per-column load.  h + m + l carries 33 bits, the fp32 wnorm
// 24; e is chosen from max |wnorm| so that |h| < 2^15.  +inf (padding, excluded copies) becomes h = -inf: the
// accumulator is -inf, the score +inf.  bias_scale[0] = E, or 0 when max |wnorm| is outside what fp16 pieces can
// carry (the kernel then keeps loading wnorm).
__global__ void __launch_bounds__(256) bias_rows_kernel(const float* __restrict__ wnorm, int Mpad,
                                                       const float* __restrict__ wmax, __half* __restrict__ Wb16,
                                                       float* __restrict__ bias_scale) {
  const float top = 0.5f * wmax[2];  // max |wnorm| / 2 over the real prototypes
  int e = 0;
  (void)frexpf(top, &e);             // top < 2^e
  e -= 15;                            // |v| / 2^e < 2^15
  if (e < -14) e = -14;
  const bool ok = e <= 15 && top == top && top < 3.0e38f;
  const float E = ok ? ldexpf(1.f, e) : 0.f;
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c == 0) bias_scale[0] = E;
  if (c >= Mpad || !ok) return;
  const float wn = wnorm[c];
  __half h, m, l;
  if (wn > 3.0e38f) {  // +inf: never a candidate
    h = __ushort_as_half((unsigned short)0xFC00);  // -inf
    m = l = __float2half_rn(0.f);
  } else {
    const float v = ldexpf(-0.5f * wn, -e);  // exact: power-of-two scaling
    h = __float2half_rn(v);
    const float r1 = v - __half2float(h);    // exact in fp32 (the pieces do not overlap)
    m = __float2half_rn(r1);
    l = __float2half_rn(r1 - __half2float(m));
  }
  __half* row = Wb16 + (int64_t)c * 64;
  row[0] = h;
  row[1] = m;
  row[2] = l;
}

// ------------------------------------------------------------------------------------------ rows
// Sequential prototype-row arithmetic of the growth step (dbgsom/BaseSom.py:641-644, :705-726,
// :824-827, :835-837): one CTA, ops in list order, a block barrier between ops.
__global__ void __launch_bounds__(256) row_ops_kernel(double* __restrict__ W, int D, const int32_t* __restrict__ ops,
                                                     int n_ops) {
  for (int o = 0; o < n_ops; ++o) {
    const int dst = ops[4 * o], a = ops[4 * o + 1], b = ops[4 * o + 2], c = ops[4 * o + 3];
    for (int d = threadIdx.x; d < D; d += 256) {
      double v = 2.0 * W[(int64_t)a * D + d] - W[(int64_t)b * D + d];
      if (c >= 0) v = (v + W[(int64_t)c * D + d]) / 2.0;
      W[(int64_t)dst * D + d] = v;
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(256) gather_rows_kernel(const float* __restrict__ X, int64_t ldx, int D,
                                                         const int64_t* __restrict__ rows, double* __restrict__ W) {
  const int r = blockIdx.x;
  const int64_t src = rows[r];
  for (int d = threadIdx.x; d < D; d += 256) W[(int64_t)r * D + d] = (double)X[src * ldx + d];
}

}  // namespace

int run_colstats(const float* X, int64_t N, int D, int64_t ldx, const float* shift, const double* weight, double* moments,
                 cudaStream_t s) {
  int64_t row_blocks = ceil_div<int64_t>(N, 4096);
  const int col_blocks = ceil_div(D, CS_COLS);
  if (row_blocks > DBGSOM_COLSTATS_PARTS) row_blocks = DBGSOM_COLSTATS_PARTS;
  if (row_blocks < 1) row_blocks = 1;
  const int64_t rows_per_block = ceil_div<int64_t>(N, row_blocks);
  const dim3 grid(col_blocks, (unsigned)row_blocks);
  if (weight)
    colstats_kernel<true><<<grid, CS_COLS * CS_ROWS, 0, s>>>(X, N, D, ldx, shift, weight, moments, rows_per_block);
  else
    colstats_kernel<false><<<grid, CS_COLS * CS_ROWS, 0, s>>>(X, N, D, ldx, shift, nullptr, moments, rows_per_block);
  DBGSOM_LAUNCH_CHECK();
  return DBGSOM_OK;
}

int run_prepare_x16(const float* X, int64_t N, int D, int64_t ldx, const float* shift, float scale, const int32_t* perm,
                    uint16_t* X16_hi, uint16_t* X16_lo, int64_t ld16, float* xnorm16, cudaStream_t s) {
  prepare_x16_kernel<<<(unsigned)ceil_div<int64_t>(N, 8), 256, 0, s>>>(
      X, N, D, ldx, shift, scale, perm, reinterpret_cast<__half*>(X16_hi), reinterpret_cast<__half*>(X16_lo), ld16, xnorm16);
  DBGSOM_LAUNCH_CHECK();
  return DBGSOM_OK;
}

int run_prepare_w(const double* W, int M, int D, const float* shift, float scale, float* W32, uint16_t* W16_hi,
                  uint16_t* W16_lo, int64_t ld16, int Mpad, const int32_t* col_of_proto, float* wnorm, double* wshift,
                  float* wmax, cudaStream_t s) {
  DBGSOM_CUDA_TRY(cudaMemsetAsync(wmax, 0, 4 * sizeof(float), s));
  if (W16_hi) {
    if (!wshift) return DBGSOM_E_BADARG;
    w_colmean_kernel<<<ceil_div(D, 32), 256, 0, s>>>(W, M, D, wshift);
    DBGSOM_LAUNCH_CHECK();
  }
  const int rows = W16_hi ? (Mpad > M ? Mpad : M) : M;
  prepare_w_kernel<<<rows, 128, 0, s>>>(W, M, D, shift, wshift, scale, W32, reinterpret_cast<__half*>(W16_hi),
                                        reinterpret_cast<__half*>(W16_lo), ld16, W16_hi ? col_of_proto : nullptr, wnorm,
                                        wmax);
  DBGSOM_LAUNCH_CHECK();
  return DBGSOM_OK;
}

int run_tile_bounds(const double* W, int M, int D, const double* wshift, float scale, const int32_t* proto_of_col,
                    const float* wnorm, int Mpad, float* out, cudaStream_t s) {
  tile_bounds_kernel<<<Mpad / 128, 256, 0, s>>>(W, M, D, wshift, scale, proto_of_col, wnorm, out);
  DBGSOM_LAUNCH_CHECK();
  return DBGSOM_OK;
}

int run_exclude_duplicates(const double* W, int M, int D, const int32_t* col_of_proto, float* wnorm,
                           unsigned long long* hash, cudaStream_t s) {
  row_hash_kernel<<<M, 128, 0, s>>>(W, M, D, hash);
  DBGSOM_LAUNCH_CHECK();
  mark_duplicates_kernel<<<ceil_div(M, 256), 256, 0, s>>>(W, M, D, hash, col_of_proto, wnorm);
  DBGSOM_LAUNCH_CHECK();
  return DBGSOM_OK;
}

int run_prepare_bias(const float* wnorm, int Mpad, const float* wmax, uint16_t* Wb16, float* bias_scale, cudaStream_t s) {
  bias_rows_kernel<<<ceil_div(Mpad, 256), 256, 0, s>>>(wnorm, Mpad, wmax, reinterpret_cast<__half*>(Wb16), bias_scale);
  DBGSOM_LAUNCH_CHECK();
  return DBGSOM_OK;
}

int run_row_ops(double* W, int D, const int32_t* ops, int n_ops, cudaStream_t s) {
  if (n_ops == 0) return DBGSOM_OK;
  row_ops_kernel<<<1, 256, 0, s>>>(W, D, ops, n_ops);
  DBGSOM_LAUNCH_CHECK();
  return DBGSOM_OK;
}

int run_gather_rows(const float* X, int64_t ldx, int D, const int64_t* rows, int n_rows, double* W, cudaStream_t s) {
  if (n_rows == 0) return DBGSOM_OK;
  gather_rows_kernel<<<n_rows, 256, 0, s>>>(X, ldx, D, rows, W);
  DBGSOM_LAUNCH_CHECK();
  return DBGSOM_OK;
}

}  // namespace dbgsom
