// Post-training passes and map maintenance on the device (SURVEY.md section 8(f) ranks 1, 2 and 4).
//
// After the epoch loop the reference runs four to five separate BMU passes with Python loops over
// the samples (dbgsom/BaseSom.py:116-127).  Here two BMU searches (top-2 on the pre-update
// prototypes, top-1 on the final reduced map) stay in HBM and these kernels reduce them:
//   node_stats_kernel   _calculate_topographic_error  dbgsom/BaseSom.py:924-953
//                       calculate_quantization_error  :904-922
//                       _calculate_node_statistics    :181-211  (hit counts, Gaussian density sums)
//   umatrix_kernel      _get_u_matrix                 :320-337  (degree-weighted mean distance of a
//                       prototype to every prototype -- quirk Q12 -- float64, direct differences like cdist)
//   label_hist_kernel   SomClassifier._label_prototypes  dbgsom/SomClassifier.py:130-152
//                       (class counts per prototype + first occurrence, which is what statistics.mode needs)
//   hops_kernel         nx.floyd_warshall_numpy(som_)  dbgsom/BaseSom.py:401  (all-pairs hop counts; the
//                       map graph has unit edges and degree <= 4, so one BFS per source replaces O(M^3))
#include "common.cuh"

namespace dbgsom {

namespace {

// ------------------------------------------------------------------------------------------ node statistics
constexpr int NS_THREADS = 256;

// out = [te_count, qe_sum, hits[M], dens_sum[M]]  (float64, atomically accumulated; zeroed by the launcher)
// WGT: every term of sample i is multiplied by weight[i] (frequency weights)
template <bool WGT>
__global__ void __launch_bounds__(NS_THREADS) node_stats_kernel(const int32_t* __restrict__ idx, int idx_stride,
                                                               const double* __restrict__ dist, int dist_stride,
                                                               int64_t N, const int32_t* __restrict__ pos, int M,
                                                               double inv_two_bw2, double norm,
                                                               const double* __restrict__ weight,
                                                               double* __restrict__ out) {
  double te = 0.0, qe = 0.0;
  double* hits = out + 2;
  double* dens = out + 2 + M;
  const int64_t stride = (int64_t)gridDim.x * NS_THREADS;
  for (int64_t i = (int64_t)blockIdx.x * NS_THREADS + threadIdx.x; i < N; i += stride) {
    const int b0 = idx[i * idx_stride];
    if ((unsigned)b0 >= (unsigned)M) continue;  // NaN row: no winner
    const double d = dist[i * dist_stride];
    const double w = WGT ? weight[i] : 1.0;
    qe += WGT ? w * d : d;
    if (idx_stride > 1) {
      const int b1 = idx[i * idx_stride + 1];
      if ((unsigned)b1 < (unsigned)M) {
        const int dx = pos[2 * b0] - pos[2 * b1], dy = pos[2 * b0 + 1] - pos[2 * b1 + 1];
        // grid distance > 1.5  <=>  squared integer distance > 2 (dbgsom/BaseSom.py:951)
        if (dx * dx + dy * dy > 2) te += w;
      }
    }
    atomicAdd(hits + b0, w);
    // (np.exp(-(d**2) / (2 * sigma**2))) / (sigma * sqrt(2 * pi))   dbgsom/BaseSom.py:205-208
    const double kd = exp(-(d * d) * inv_two_bw2) * norm;
    atomicAdd(dens + b0, WGT ? w * kd : kd);
  }
  te = warp_sum(te);
  qe = warp_sum(qe);
  __shared__ double sh[2][NS_THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) {
    sh[0][warp] = te;
    sh[1][warp] = qe;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int w = 0; w < NS_THREADS / 32; ++w) {
      a += sh[0][w];
      b += sh[1][w];
    }
    atomicAdd(out + 0, a);
    atomicAdd(out + 1, b);
  }
}

// ------------------------------------------------------------------------------------------ class histogram
// weight != NULL: first occurrences over the samples with weight > 0 only.  counts == NULL: first occurrences only (the
// weighted counts are summed per winner in a fixed order by the segment kernel of accumulate.cu)
__global__ void __launch_bounds__(NS_THREADS) label_hist_kernel(const int32_t* __restrict__ idx, int idx_stride,
                                                               const int32_t* __restrict__ labels,
                                                               const double* __restrict__ weight, int64_t N,
                                                               int64_t sample_offset, int M, int n_classes,
                                                               int32_t* __restrict__ counts,
                                                               long long* __restrict__ first) {
  const int64_t stride = (int64_t)gridDim.x * NS_THREADS;
  for (int64_t i = (int64_t)blockIdx.x * NS_THREADS + threadIdx.x; i < N; i += stride) {
    const int b = idx[i * idx_stride];
    const int y = labels[i];
    if ((unsigned)b >= (unsigned)M || (unsigned)y >= (unsigned)n_classes) continue;
    if (weight && !(weight[i] > 0.0)) continue;
    const int64_t cell = (int64_t)b * n_classes + y;
    if (counts) atomicAdd(counts + cell, 1);
    atomicMin(first + cell, (long long)(sample_offset + i));
  }
}

__global__ void fill_i64_kernel(long long* p, int64_t n, long long v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// ------------------------------------------------------------------------------------------ u-matrix
// out[i] += sum_{j in tile} colw[j] * ||W[i] - W[j]||_2 ; CTA = 64 x 64 pairs, thread = 4 x 4 pairs,
// k streamed through shared memory 16 columns at a time.  float64 throughout.
constexpr int UM_TILE = 64;
constexpr int UM_K = 16;
__global__ void __launch_bounds__(256) umatrix_kernel(const double* __restrict__ W, int M, int D, int64_t ldw,
                                                     const double* __restrict__ colw, double* __restrict__ out) {
  __shared__ double As[UM_K][UM_TILE + 2];
  __shared__ double Bs[UM_K][UM_TILE + 2];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int i0 = blockIdx.y * UM_TILE, j0 = blockIdx.x * UM_TILE;
  double acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
  const int lr = threadIdx.x >> 2;        // row of the tile this thread loads
  const int lk = (threadIdx.x & 3) * 4;   // first of its 4 columns
  for (int k0 = 0; k0 < D; k0 += UM_K) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int k = k0 + lk + q;
      const int ri = i0 + lr, rj = j0 + lr;
      As[lk + q][lr] = (ri < M && k < D) ? W[(int64_t)ri * ldw + k] : 0.0;
      Bs[lk + q][lr] = (rj < M && k < D) ? W[(int64_t)rj * ldw + k] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < UM_K; ++k) {
      double a[4], b[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        a[q] = As[k][ty * 4 + q];
        b[q] = Bs[k][tx * 4 + q];
      }
#pragma unroll
      for (int p = 0; p < 4; ++p)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const double t = a[p] - b[q];
          acc[p][q] = fma(t, t, acc[p][q]);
        }
    }
    __syncthreads();
  }
  // weighted row sums over this tile's 64 columns: 16 threads (tx) share a row
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    double s = 0.0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int j = j0 + tx * 4 + q;
      if (j < M) s += colw[j] * sqrt(acc[p][q]);
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(kFullMask, s, o);
    const int i = i0 + ty * 4 + p;
    if (tx == 0 && i < M) atomicAdd(out + i, s);
  }
}

// ------------------------------------------------------------------------------------------ hop matrix
// One CTA per source node: level-synchronous BFS over the adjacency table adj[M][4] (-1 = no edge).
// Shared memory: dist int32 [M] + two frontier queues uint16 [M] each (M <= 28000).
constexpr int HOP_THREADS = 256;
constexpr int HOP_MAX_M = 28000;
__global__ void __launch_bounds__(HOP_THREADS) hops_kernel(const int32_t* __restrict__ adj, int M,
                                                          uint16_t* __restrict__ hop, int64_t ldh) {
  extern __shared__ __align__(16) uint8_t hop_smem[];
  int32_t* dist = reinterpret_cast<int32_t*>(hop_smem);
  uint16_t* q0 = reinterpret_cast<uint16_t*>(dist + M);
  uint16_t* q1 = q0 + M;
  __shared__ int n_next;
  for (int src = blockIdx.x; src < M; src += gridDim.x) {
    for (int i = threadIdx.x; i < M; i += HOP_THREADS) dist[i] = 0xFFFF;
    __syncthreads();
    if (threadIdx.x == 0) {
      dist[src] = 0;
      q0[0] = (uint16_t)src;
      n_next = 0;
    }
    __syncthreads();
    uint16_t *cur = q0, *nxt = q1;
    int n_cur = 1;
    for (int level = 1; n_cur > 0; ++level) {
      for (int f = threadIdx.x; f < n_cur; f += HOP_THREADS) {
        const int u = cur[f];
        const int4 nb = *reinterpret_cast<const int4*>(adj + 4 * (int64_t)u);
        const int v[4] = {nb.x, nb.y, nb.z, nb.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (v[e] >= 0 && atomicCAS(&dist[v[e]], 0xFFFF, level) == 0xFFFF) nxt[atomicAdd(&n_next, 1)] = (uint16_t)v[e];
        }
      }
      __syncthreads();
      n_cur = n_next;
      __syncthreads();
      if (threadIdx.x == 0) n_next = 0;
      uint16_t* t = cur;
      cur = nxt;
      nxt = t;
      // the reset of n_next is ordered before the next level's pushes by the barrier at the end of that level's
      // predecessor loop: pushes only happen after every thread passed the barrier above
      __syncthreads();
    }
    for (int i = threadIdx.x; i < M; i += HOP_THREADS) hop[(int64_t)src * ldh + i] = (uint16_t)dist[i];
    __syncthreads();
  }
}

}  // namespace

int run_node_stats(const int32_t* idx, int idx_stride, const double* dist, int dist_stride, int64_t N,
                   const int32_t* pos, int M, double bandwidth, const double* weight, double* out, cudaStream_t s) {
  DBGSOM_CUDA_TRY(cudaMemsetAsync(out, 0, (size_t)(2 + 2 * (int64_t)M) * sizeof(double), s));
  int64_t blocks = ceil_div<int64_t>(N, NS_THREADS * 8);
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  const double inv_two_bw2 = 1.0 / (2.0 * bandwidth * bandwidth);
  const double norm = 1.0 / (bandwidth * 2.5066282746310002);  // sqrt(2 pi)
  if (weight)
    node_stats_kernel<true><<<(unsigned)blocks, NS_THREADS, 0, s>>>(idx, idx_stride, dist, dist_stride, N, pos, M,
                                                                   inv_two_bw2, norm, weight, out);
  else
    node_stats_kernel<false><<<(unsigned)blocks, NS_THREADS, 0, s>>>(idx, idx_stride, dist, dist_stride, N, pos, M,
                                                                    inv_two_bw2, norm, nullptr, out);
  DBGSOM_LAUNCH_CHECK();
  return DBGSOM_OK;
}

// weight != NULL: first occurrences among the samples with weight > 0 only; counts may be NULL (see label_hist_kernel)
int run_label_hist(const int32_t* idx, int idx_stride, const int32_t* labels, const double* weight, int64_t N,
                   int64_t sample_offset, int M, int n_classes, int32_t* counts, int64_t* first, cudaStream_t s) {
  const int64_t cells = (int64_t)M * n_classes;
  if (counts) DBGSOM_CUDA_TRY(cudaMemsetAsync(counts, 0, (size_t)cells * sizeof(int32_t), s));
  fill_i64_kernel<<<(unsigned)ceil_div<int64_t>(cells, 256), 256, 0, s>>>(reinterpret_cast<long long*>(first), cells,
                                                                         0x7fffffffffffffffLL);
  DBGSOM_LAUNCH_CHECK();
  int64_t blocks = ceil_div<int64_t>(N, NS_THREADS * 8);
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  label_hist_kernel<<<(unsigned)blocks, NS_THREADS, 0, s>>>(idx, idx_stride, labels, weight, N, sample_offset, M,
                                                           n_classes, counts, reinterpret_cast<long long*>(first));
  DBGSOM_LAUNCH_CHECK();
  return DBGSOM_OK;
}

int run_umatrix(const double* W, int M, int D, int64_t ldw, const double* colw, double* out, cudaStream_t s) {
  DBGSOM_CUDA_TRY(cudaMemsetAsync(out, 0, (size_t)M * sizeof(double), s));
  const unsigned t = (unsigned)ceil_div(M, UM_TILE);
  umatrix_kernel<<<dim3(t, t), 256, 0, s>>>(W, M, D, ldw, colw, out);
  DBGSOM_LAUNCH_CHECK();
  return DBGSOM_OK;
}

int run_hops(const int32_t* adj, int M, uint16_t* hop, int64_t ldh, cudaStream_t s) {
  if (M > HOP_MAX_M) return DBGSOM_E_UNSUPPORTED;
  const size_t smem = (size_t)M * 4 + 2 * (size_t)M * 2 + 16;
  DBGSOM_CUDA_TRY(cudaFuncSetAttribute(hops_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = (int)((220 * 1024) / (smem + 1024));
  if (per_sm > 8) per_sm = 8;
  if (per_sm < 1) per_sm = 1;
  int blocks = 148 * per_sm;
  if (blocks > M) blocks = M;
  hops_kernel<<<blocks, HOP_THREADS, smem, s>>>(adj, M, hop, ldh);
  DBGSOM_LAUNCH_CHECK();
  return DBGSOM_OK;
}

}  // namespace dbgsom
