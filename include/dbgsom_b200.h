/*
 * dbgsom_b200 -- C ABI of the B200-native batch-SOM training epoch.
 *
 * The reference (SandroMartens/DBGSOM) is pure Python and has no FFI of its own; the
 * boundary it offers is a set of numpy-in / numpy-out methods on `BaseSom`
 * (dbgsom/BaseSom.py).  Each entry point below replaces one of those methods (cited per
 * function) and is what a ctypes binding inside that class would call; see INTEGRATION.md
 * for the stub.  Conventions:
 *
 *   - every pointer named d_* is a DEVICE pointer owned by the caller (the Python host code
 *     takes them from torch tensors); nothing here allocates or frees device memory;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and the call
 *     returns without synchronising unless stated otherwise;
 *   - every function returns 0 on success, a negative DBGSOM_E_* code for argument errors,
 *     or a positive cudaError_t; nothing throws; the library keeps no global state besides
 *     cached device attributes and the resolved cuTensorMapEncodeTiled entry point;
 *   - matrices are row-major; `ld*` are leading dimensions in ELEMENTS;
 *   - sizes: N samples, D features, M prototypes ("neurons");
 *   - d_weight (the *_weighted entry points): float64 [N] frequency weights of the samples (sample_weight of
 *     fit), finite and >= 0; NULL = every weight 1, which is exactly the unweighted entry point.  A sample of
 *     weight w counts like w copies of it in every sum.  This is unrelated to the per-sample similarity
 *     k_i of K2, which the reference calls "sample_weights".
 *
 * Data layout in HBM (see DESIGN.md):
 *   X     float32 [N, ldx]      master copy of the samples (read by the update pass)
 *   X16   float16 [N, ld16] x2  shadow (X - shift) * scale split as hi + lo (lo only for the
 *                               three-pass search), ld16 = D rounded up to 64, pad = 0
 *   W     float64 [Mcap, D]     master prototypes (neuron order = node insertion order)
 *   W32   float32 [Mcap, D]     rounded copy used by the streaming kernels
 *   W16   float16 [Mpad, ld16] x2  shadow (W - mean_j W) * scale as hi + lo, Mpad = M rounded up to 256
 *   hop   uint16  [M, ldh]      all-pairs hop counts of the map graph, 0xFFFF = unreachable
 *   part  float64 [M*D + 3M]    per-epoch partial sums  [ Sk | sk | n | E ]  (one all-reduce)
 */
#ifndef DBGSOM_B200_H
#define DBGSOM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DBGSOM_ABI_VERSION 10

#define DBGSOM_OK 0
#define DBGSOM_E_BADARG (-1)      /* null pointer, non-positive size, bad enum             */
#define DBGSOM_E_WORKSPACE (-2)   /* workspace smaller than dbgsom_*_workspace_bytes says  */
#define DBGSOM_E_UNSUPPORTED (-3) /* shape outside what the kernel handles (e.g. D too big)*/
#define DBGSOM_E_DRIVER (-4)      /* cuTensorMapEncodeTiled unavailable / failed           */
#define DBGSOM_E_NOT_SM100 (-5)   /* device is not compute capability 10.x                 */

#define DBGSOM_MAX_CAND 8         /* candidate slots per sample and rank                   */
#define DBGSOM_CAND_OVERFLOW 255  /* cand_count value: more near-ties than slots           */
#define DBGSOM_HOP_INF 0xFFFFu

/* BMU candidate-search back ends (both are followed by the same exact re-score). */
#define DBGSOM_BMU_SIMT 0   /* fp32 CUDA cores, direct differences                         */
#define DBGSOM_BMU_TENSOR 1 /* fp16 tcgen05.mma, TMEM accumulators, TMA-fed                */

int dbgsom_abi_version(void);
/* Human-readable text for a status returned by any function below. */
const char* dbgsom_status_string(int status);
/* 0 if device `device` can run the kernels (compute capability 10.x), else DBGSOM_E_NOT_SM100. */
int dbgsom_check_device(int device);

/* ------------------------------------------------------------------------------------------
 * K4  column statistics (once per fit)
 * replaces  np.var(data, axis=0).sum()           dbgsom/BaseSom.py:363
 *           np.std(data, axis=0, ddof=1)         dbgsom/BaseSom.py:380
 * d_moments is [DBGSOM_COLSTATS_PARTS][2D+1]; part r covers a fixed block of rows:
 * part[0:D] = sum_i (x_id - c_d),  part[D:2D] = sum_i (x_id - c_d)^2 in float64,
 * part[2D] = max(part[2D], max_id |x_id - c_d|), with c = d_shift_row (float32 [D],
 * device; any data row works, all ranks must use the same one).  The caller zeroes d_moments,
 * adds the parts in order (max for the last entry; a fixed order makes the result the same on
 * every run), all-reduces the sum across GPUs when sharded and finishes the scalars on the host.
 */
#define DBGSOM_COLSTATS_PARTS 256
int dbgsom_colstats(const float* d_X, int64_t N, int D, int64_t ldx, const float* d_shift_row,
                    double* d_moments, void* stream);
/* Same with frequency weights: part[0:D] = sum_i w_i (x_id - c_d), part[D:2D] = sum_i w_i (x_id - c_d)^2; the
 * maximum stays over ALL rows (zero-weight rows too: every row goes through the fp16 shadow it scales).  The
 * caller divides by sum_i w_i instead of N. */
int dbgsom_colstats_weighted(const float* d_X, int64_t N, int D, int64_t ldx, const float* d_shift_row,
                             const double* d_weight, double* d_moments, void* stream);

/* ------------------------------------------------------------------------------------------
 * fp16 shadows for the tensor-core BMU search (X once per fit, W once per epoch)
 *
 * x' = (x - shift) * scale is split as hi = fp16(x'), lo = fp16(x' - hi); d_X16_lo may be NULL
 * when only the single-pass search is used.  d_xnorm16[i] = ||x'_i||_2 (for the error bound).
 */
int dbgsom_prepare_x16(const float* d_X, int64_t N, int D, int64_t ldx, const float* d_shift /*[D]*/,
                       float scale, uint16_t* d_X16_hi, uint16_t* d_X16_lo, int64_t ld16,
                       float* d_xnorm16 /*[N]*/, void* stream);

/* Same, with the shadow rows in a caller-given order: shadow row p is built from sample d_perm[p] (a permutation of
 * 0..N-1, e.g. the samples grouped by winner that dbgsom_accumulate leaves in its workspace, see
 * dbgsom_accumulate_perm_offset); d_xnorm16 stays indexed by SAMPLE.  Pass the permutation to the search as
 * dbgsom_bmu_args.d_row_perm. */
int dbgsom_prepare_x16_sorted(const float* d_X, int64_t N, int D, int64_t ldx, const float* d_shift, float scale,
                              const int32_t* d_perm, uint16_t* d_X16_hi, uint16_t* d_X16_lo, int64_t ld16,
                              float* d_xnorm16, void* stream);

/* W (float64 master) -> W32, and optionally the fp16 shadow of the tensor back end.
 * With c = mean_j W[j,:] (written to d_wshift, float64 [D]), u_j = (w_j - c) * scale and
 * v = (c - shift) * scale:  W16_hi + W16_lo ~= u_j,  d_wnorm[j] = ||u_j||^2 + 2 u_j.v, so that
 * d_wnorm[j] - 2 x'.u_j equals ||x' - (w_j - shift) * scale||^2 up to a per-sample constant.
 * d_W16_hi/lo, d_wnorm, d_wshift may be NULL (SIMT back end).  Shadow row and wnorm entry of
 * prototype j are stored at position d_col_of_proto[j] (a permutation of [0, Mpad); NULL = identity):
 * the tensor kernel visits prototypes in shadow order and a pseudo-random order keeps the number
 * of running-minimum updates per sample at ~ln(M) even on a smooth map.  The Mpad - M padding
 * positions are zeroed and their wnorm set to +inf so they can never win.  d_wmax receives
 * { max_j ||u_j||_2, max_j ||w_j||_2, max_j |wnorm_j|, max_jd |u_jd| }: the first three feed the
 * candidate error bounds; if the last reaches the fp16 range (65504) the shadow was clamped and
 * the caller must use the SIMT back end for these prototypes.
 */
int dbgsom_prepare_w(const double* d_W, int M, int D, const float* d_shift, float scale, float* d_W32,
                     uint16_t* d_W16_hi, uint16_t* d_W16_lo, int64_t ld16, int Mpad,
                     const int32_t* d_col_of_proto /*[Mpad] or NULL*/, float* d_wnorm /*[Mpad]*/,
                     double* d_wshift /*[D]*/, float* d_wmax /*[4]*/, void* stream);

/* Optional, after dbgsom_prepare_w and before a top-1 (n_bmu = 1) tensor search: sets wnorm to +inf for every
 * prototype that equals a LOWER-indexed prototype element by element.  The reference gives exact distance ties
 * to the lowest index (sklearn/utils/_heap.pyx:46), so such a copy can never be the answer of a top-1 search;
 * with the copies out of the search the epilogue may keep equally scored prototypes in any order
 * (dbgsom_bmu_args.ties_any = 1), which removes most of its work on collapsed maps (thousands of near-identical
 * prototypes).  Do not use it for n_bmu = 2, where a copy is the legitimate second winner.
 * d_hash: scratch, M 64-bit words. */
int dbgsom_exclude_duplicates(const double* d_W, int M, int D, const int32_t* d_col_of_proto /*[M..] or NULL*/,
                              float* d_wnorm, uint64_t* d_hash, void* stream);

/* Optional, after dbgsom_prepare_w (and dbgsom_exclude_duplicates): d_tile_bound[2 q], [2 q + 1] = max ||u_j||_2 and
 * max |wnorm_j| over the prototypes in shadow columns [128 q, 128 q + 128), rounded up; padding columns and prototypes
 * taken out of the search (wnorm = +inf) do not count.  d_proto_of_col as in dbgsom_bmu_args (NULL = identity),
 * d_wshift and scale as written / given to dbgsom_prepare_w; Mpad a multiple of 128.  Passed on in
 * dbgsom_bmu_args.d_tile_bound it lets the candidate search for D > 256 bound the rounding error of a score by the
 * norms of its own column tile. */
int dbgsom_tile_bounds(const double* d_W, int M, int D, const double* d_wshift /*[D]*/, float scale,
                       const int32_t* d_proto_of_col /*[Mpad] or NULL*/, const float* d_wnorm /*[Mpad]*/, int Mpad,
                       float* d_tile_bound /*[Mpad / 128, 2]*/, void* stream);

/* Optional, after dbgsom_prepare_w (and dbgsom_exclude_duplicates): wnorm as an MMA operand.  Writes three fp16
 * pieces of -wnorm / (2 E) into the first three columns of d_Wb16[c, 0:64] (c = shadow row; the other columns must
 * be zero and are not touched) and E, a power of two chosen from max |wnorm|, into d_bias_scale[0] (0 = the values
 * do not fit fp16 pieces: the search then keeps loading wnorm).  With dbgsom_bmu_args.d_Wb16 / d_bias_scale set, the
 * CTA-pair form of the tensor search ends every output tile with one extra k-step (A = E in three columns), so its
 * epilogue reads scores straight from the accumulator. */
int dbgsom_prepare_bias(const float* d_wnorm, int Mpad, const float* d_wmax, uint16_t* d_Wb16 /*[Mpad, 64]*/,
                        float* d_bias_scale /*[1]*/, void* stream);

/* ------------------------------------------------------------------------------------------
 * K1  best-matching-unit search
 * replaces  BaseSom._get_winning_neurons(data, n_bmu)   dbgsom/BaseSom.py:446-464
 *           (sklearn NearestNeighbors(n_neighbors=n_bmu).fit(W).kneighbors(X))
 *
 * Two stages.  (1) candidate search over all M prototypes with an approximate score and a
 * per-sample error bound: every prototype whose score is within the bound of the n_bmu-th best
 * is kept (up to DBGSOM_MAX_CAND, else the sample is flagged DBGSOM_CAND_OVERFLOW).
 * (2) exact re-score in float64 of the kept candidates; ties go to the lowest index like
 * sklearn's heap.  A flagged sample has more than DBGSOM_MAX_CAND prototypes inside its bound:
 * if the bound is below `tie_rel` (relative, squared distance; default 1e-6 = the parity gate of
 * BASELINE.json) the best approximate candidate is returned, otherwise -- or always when
 * strict != 0 -- the sample is re-scored against all M prototypes in float64.
 * Results therefore equal the float64 brute-force search wherever best and second-best squared
 * distance differ by more than max(~1e-12, tie_rel) relative.
 *
 * Tensor back end: n_pass = 1 uses X16_hi . W16_hi (fp16 inputs, error ~2^-11, only useful when
 * prototypes are well separated); n_pass = 3 adds the hi.lo and lo.hi products (error ~2^-21).
 */
typedef struct dbgsom_bmu_args {
  /* samples */
  const float* d_X;        /* [N, ldx] */
  const uint16_t* d_X16_hi; /* [N, ld16] fp16 shadow; may be NULL for DBGSOM_BMU_SIMT */
  const uint16_t* d_X16_lo; /* [N, ld16] residual shadow; needed for n_pass = 3 */
  const float* d_xnorm16;  /* [N] ||x'||_2; may be NULL for DBGSOM_BMU_SIMT */
  int64_t N;
  int32_t D;
  int64_t ldx;
  int64_t ld16;
  /* prototypes */
  const double* d_W;       /* [M, D] float64 master (exact re-score) */
  const float* d_W32;      /* [M, D] */
  const uint16_t* d_W16_hi; /* [Mpad, ld16]; may be NULL for DBGSOM_BMU_SIMT */
  const uint16_t* d_W16_lo; /* [Mpad, ld16]; needed for n_pass = 3 */
  const float* d_wnorm;    /* [Mpad]; may be NULL for DBGSOM_BMU_SIMT */
  const uint16_t* d_Wb16;  /* [Mpad, 64] from dbgsom_prepare_bias, or NULL (used by the classic CTA-pair search for
                              D <= 256 and by the FLAG pass of the selective search for D <= 128) */
  const float* d_bias_scale; /* [1] from dbgsom_prepare_bias, or NULL */
  const float* d_wmax;     /* [4] from dbgsom_prepare_w */
  const int32_t* d_proto_of_col; /* [Mpad] prototype index stored in shadow row c (tensor back end;
                              the inverse of the map given to dbgsom_prepare_w; entries >= M are padding) */
  float scale;             /* the scale both shadows were built with */
  int32_t M;
  int32_t Mpad;
  int32_t proto_stride;    /* optional hint, 0 = none: a value s > 0 promises d_proto_of_col[c] == (c * s) % Mpad
                              for every c (s coprime to Mpad, Mpad < 65536); the candidate search then evaluates
                              prototype indices in registers instead of loading them */
  int32_t ties_any;        /* 1: prototypes with EQUAL approximate scores may be kept in any order (n_bmu = 1
                              only, and only after dbgsom_exclude_duplicates); 0: ordered by prototype index, so
                              the lowest index among exact copies always survives */
  /* request */
  int32_t n_bmu;           /* 1 or 2 */
  int32_t backend;         /* DBGSOM_BMU_SIMT / DBGSOM_BMU_TENSOR */
  int32_t n_pass;          /* tensor back end: 1 or 3 */
  float bound_scale;       /* multiplies the rounding bound of the tensor back end; 1.0 = worst-case
                              (Cauchy-Schwarz) bound; <= 0 selects the calibrated default (0.25 for
                              one pass, 0.0625 for three, see csrc/common.cuh) */
  float tie_rel;           /* see above; <= 0 selects 1e-6 */
  int32_t strict;          /* 1: flagged samples are always re-scored against all prototypes, and the fp32
                              accumulation term of the tensor bound grows linearly (default: with the square
                              root) with the accumulation chain for D > 256 (csrc/common.cuh tensor_acc_coef) */
  int32_t want_dist;       /* 0: winners only (training epoch); 1: also exact distances */
  /* outputs */
  int32_t* d_idx;          /* [N, n_bmu] winners, ascending distance */
  double* d_dist;          /* [N, n_bmu] Euclidean distances (want_dist=1), else may be NULL */
  int64_t* d_stats;        /* optional [8], atomically incremented: #samples with more candidates than
                              n_bmu, #flagged samples, #candidates re-scored, #full re-scores, and by the selective
                              search (below) #(row-tile pair, column tile) products refined, #row-tile pairs,
                              column tiles per row-tile pair; [7] reserved */
  /* scratch */
  void* d_workspace;
  size_t workspace_bytes;
  /* sorted sample order + selective search (tensor back end, n_bmu = 1; all optional, zero = off).
   * d_row_perm: the fp16 shadows were built by dbgsom_prepare_x16_sorted, i.e. shadow row p belongs to sample
   * d_row_perm[p]; every per-sample output (d_idx, the candidate table) is written at the sample's own index.
   * select = DBGSOM_SELECT_FLAG runs ONE fp16 pass (bound of n_pass = 1) over all prototypes and only records, per
   * pair of 128-row tiles, which column tiles of `select_granule` prototypes hold a score within the one-pass bound
   * of the smallest one-pass score of any of its rows (bit c of d_tile_mask[pair], OR-ed in: zero the masks first).
   * select = DBGSOM_SELECT_REFINE runs the three-pass candidate search of n_pass = 3 over exactly those column tiles.
   * The exact winner's one-pass score is within twice the one-pass error bound of the row's best one-pass score, so
   * its column tile is always refined; with the rows sorted by their previous winner and the shadow columns laid
   * out in map patches a row-tile pair touches few column tiles. */
  const int32_t* d_row_perm;      /* [N] or NULL */
  uint64_t* d_tile_mask;          /* [ceil(ceil(N / 128) / 2)] */
  const float* d_tile_bound;      /* optional, [Mpad / 128, 2] from dbgsom_tile_bounds: max ||u_j|| and max |wnorm_j| per 128
                                     shadow columns.  The candidate search for D > 256 (n_bmu = 1) then bounds the rounding
                                     error of a score with the maxima of ITS column tile (floored at 1/8 of the map-wide
                                     ones) instead of the map-wide maxima; NULL = map-wide bound everywhere */
  int32_t select;                 /* DBGSOM_SELECT_OFF / _FLAG / _REFINE */
  int32_t select_granule;         /* 64 or 128 prototypes per mask bit; Mpad / granule <= 64 */
} dbgsom_bmu_args;

#define DBGSOM_SELECT_OFF 0
#define DBGSOM_SELECT_FLAG 1
#define DBGSOM_SELECT_REFINE 2

/* 1 if the selective search (select != 0) is implemented for these shapes (D <= 256 after padding, at least one
 * row tile per SM, Mpad <= 4096 and Mpad / select_granule <= 64, n_bmu = 1), else 0. */
int dbgsom_bmu_select_supported(int64_t N, int64_t ld16, int32_t Mpad, int32_t n_bmu, int32_t select_granule);

size_t dbgsom_bmu_workspace_bytes(int64_t N, int32_t n_bmu);
int dbgsom_bmu(const dbgsom_bmu_args* args, void* stream);
/* The two stages of dbgsom_bmu as separate calls (same arguments): candidate search writes the
 * candidate table into the workspace and provisional winners into d_idx; resolve re-scores. */
int dbgsom_bmu_candidates(const dbgsom_bmu_args* args, void* stream);
int dbgsom_bmu_resolve(const dbgsom_bmu_args* args, void* stream);

/* ------------------------------------------------------------------------------------------
 * K2  sample weights + per-BMU segmented accumulation
 * replaces  _calculate_exp_similarity            dbgsom/BaseSom.py:533-538
 *           argsort/unique + numba_voronoi_set_centers   :488-497, :1028-1055  (numerators/denominators)
 *           neuron_activations                   :500-503
 *           numba_quantization_error             :1058-1073
 *
 * For every sample i with winner b = d_bmu[i]:  d_i = ||x_i - w_b||_2 (float64, direct differences),
 * k_i = 1 - sqrt(1 - exp(-d_i^2 / total_variance))  (float64, the reference's expression),
 *   Sk[b,:] += k_i x_i,  sk[b] += k_i,  n[b] += 1,  E[b] += d_i.
 * d_part is the contiguous float64 buffer [Sk (M*D) | sk (M) | n (M) | E (M)]; the call zeroes it
 * first.  Samples are bucketed by winner (counting sort) and each bucket is streamed once with
 * its prototype in registers, so X is read exactly once.
 * If d_labels != NULL, d_class_hist [M, n_classes] (int32, zeroed by the call) receives the class
 * histogram per winner (entropy growth criterion, dbgsom/BaseSom.py:547-551).
 */
typedef struct dbgsom_accumulate_args {
  const float* d_X;
  int64_t N;
  int32_t D;
  int64_t ldx;
  const int32_t* d_bmu;    /* [N] (stride 1) */
  const double* d_W;       /* [M, D] float64 master prototypes */
  int32_t M;
  double inv_total_variance;
  double* d_part;          /* [M*D + 3M] */
  const int32_t* d_labels; /* [N] or NULL */
  int32_t n_classes;
  int32_t* d_class_hist;   /* [M, n_classes] or NULL */
  void* d_workspace;
  size_t workspace_bytes;
} dbgsom_accumulate_args;

size_t dbgsom_accumulate_workspace_bytes(int64_t N, int32_t M, int32_t D);
/* Byte offset, inside the workspace of dbgsom_accumulate(N, M), of the int32 [N] sample permutation grouped by
 * winner (ascending winner index) that the call leaves behind.  For M <= 24576 the samples of a winner are in
 * ascending sample index and the call's sums are the same on every run; above that the samples of a winner are
 * in the order the scatter's atomics hand out, which varies between runs, and so do the last bits of the sums. */
size_t dbgsom_accumulate_perm_offset(int64_t N, int32_t M);
int dbgsom_accumulate(const dbgsom_accumulate_args* args, void* stream);
/* Same with frequency weights w_i = d_weight[i]:  Sk[b,:] += w_i k_i x_i,  sk[b] += w_i k_i,  n[b] += w_i,
 * E[b] += w_i d_i.  A neuron is live iff n > 0: one that wins only zero-weight samples is dead.  The samples are
 * still bucketed by integer count; the weight of each row is read with the row.  With d_labels, the class
 * histogram per winner is summed as float64 weights into d_class_hist_w [M, n_classes] (every cell written;
 * args->d_class_hist is not used), in a fixed order per winner, so it is the same on every run for M <= 24576
 * like the other sums.  d_weight == NULL is dbgsom_accumulate (int32 d_class_hist, d_class_hist_w unused). */
int dbgsom_accumulate_weighted(const dbgsom_accumulate_args* args, const double* d_weight, double* d_class_hist_w,
                               void* stream);

/* ------------------------------------------------------------------------------------------
 * K3  neighbourhood smoothing
 * replaces  _calculate_gaussian_neighborhood     dbgsom/BaseSom.py:525-531
 *           _update_weights steps 4-5            dbgsom/BaseSom.py:509-523
 *
 * centres C'[r] = Sk[j]/sk[j] for the r-th live neuron j (pack_rows=1, reference behaviour: rows
 * are packed, SURVEY.md quirk Q1) or C'[j] = Sk[j]/sk[j] (pack_rows=0);
 * W_out[i,:] = sum_j H_ij n_j C'[j,:] / sum_j H_ij n_j   with  H_ij = d_kernel_lut[hop_ij];
 * d_change[0] = sum_i ||W_in[i,:] - W_out[i,:]||_2   (the call zeroes it first).
 * d_kernel_lut [lut_len] float64 holds exp(-h^2 / (2 sigma^2)) for h = 0..lut_len-1, computed by
 * the host with the same numpy expression as the reference; hop 0xFFFF or >= lut_len gives H = 0.
 * Both sums run over the neurons with n_j > 0 only (the others contribute exact zeros).
 * All arithmetic is float64.
 */
typedef struct dbgsom_smooth_args {
  const double* d_part;      /* [M*D + 3M] (after the all-reduce when sharded) */
  const uint16_t* d_hop;     /* [M, ldh] */
  int64_t ldh;
  const double* d_kernel_lut;
  int32_t lut_len;
  int32_t M;
  int32_t D;
  int32_t pack_rows;
  const double* d_W_in;      /* [M, D] */
  double* d_W_out;           /* [M, D] (must not alias d_W_in) */
  double* d_change;          /* [1] */
  void* d_workspace;
  size_t workspace_bytes;
  int32_t row_begin;         /* rows [row_begin, row_end) of W_out are written and summed into d_change; */
  int32_t row_end;           /* row_end <= row_begin means all M rows.  Sharded maps: every rank takes a row range
                                and all-gathers W_out (the sums over the neurons are not split). */
} dbgsom_smooth_args;

size_t dbgsom_smooth_workspace_bytes(int32_t M, int32_t D);
int dbgsom_smooth(const dbgsom_smooth_args* args, void* stream);

/* ------------------------------------------------------------------------------------------
 * growth support: prototype rows of inserted neurons
 * replaces  the weight arithmetic of _insert_neuron_1p/_2p/_3p  dbgsom/BaseSom.py:641-644, :705-726,
 *           :824-827, :835-837  (2*W[a] - W[b], optionally averaged with W[c]); ops are applied
 *           sequentially in list order (a later op may read a row written by an earlier one).
 * d_ops is int32 [n_ops, 4] = (dst, a, b, c) with c = -1 for the two-term form.
 */
int dbgsom_apply_row_ops(double* d_W, int D, const int32_t* d_ops, int n_ops, void* stream);

/* W[r,:] = X[rows[r],:] (float32 -> float64) -- the start prototypes, dbgsom/BaseSom.py:423-430 */
int dbgsom_gather_rows(const float* d_X, int64_t ldx, int D, const int64_t* d_rows, int n_rows,
                       double* d_W, void* stream);

/* ------------------------------------------------------------------------------------------
 * post-training passes (SURVEY.md section 8(f) rank 1): the reference runs four to five separate BMU
 * passes with Python loops over the samples after the epoch loop (dbgsom/BaseSom.py:116-127); here
 * the winners / distances of two device BMU searches stay in HBM and are reduced by these calls.
 *
 * dbgsom_node_stats  replaces  _calculate_topographic_error  dbgsom/BaseSom.py:924-953
 *                              calculate_quantization_error  dbgsom/BaseSom.py:904-922
 *                              _calculate_node_statistics    dbgsom/BaseSom.py:181-211
 *   d_idx [N, idx_stride] winners (column 0 = BMU, column 1 = second BMU when idx_stride >= 2),
 *   d_dist [N, dist_stride] distances (column 0), d_pos [M, 2] grid coordinates of the neurons.
 *   d_out float64 [2 + 2M] = [#samples whose two BMUs are more than 1.5 apart on the grid,
 *   sum of BMU distances, hit count per neuron, sum of exp(-d^2 / (2 bw^2)) / (bw sqrt(2 pi)) per neuron];
 *   zeroed by the call.
 */
int dbgsom_node_stats(const int32_t* d_idx, int32_t idx_stride, const double* d_dist, int32_t dist_stride,
                      int64_t N, const int32_t* d_pos, int32_t M, double bandwidth, double* d_out, void* stream);
/* Same with frequency weights: every sample's term (topographic-error indicator, distance, hit, density term) is
 * multiplied by d_weight[i]; the caller divides the first two by sum_i w_i. */
int dbgsom_node_stats_weighted(const int32_t* d_idx, int32_t idx_stride, const double* d_dist, int32_t dist_stride,
                               int64_t N, const int32_t* d_pos, int32_t M, double bandwidth, const double* d_weight,
                               double* d_out, void* stream);

/* replaces  BaseSom._get_u_matrix  dbgsom/BaseSom.py:320-337:
 * d_out[i] = sum_j d_colw[j] * ||W[i,:] - W[j,:]||_2  (float64, direct differences like scipy cdist);
 * the caller passes d_colw[j] = degree(j) / sum of degrees (quirk Q12).  d_out is zeroed by the call. */
int dbgsom_umatrix(const double* d_W, int32_t M, int32_t D, int64_t ldw, const double* d_colw, double* d_out,
                   void* stream);

/* replaces  SomClassifier._label_prototypes  dbgsom/SomClassifier.py:130-152 (the per-neuron class
 * statistics it loops over the samples for): d_counts int32 [M, n_classes] class histogram per winner,
 * d_first int64 [M, n_classes] smallest global sample index (sample_offset + row) per cell, INT64_MAX if
 * empty -- statistics.mode returns the most frequent class met first.  Both are initialised by the call. */
int dbgsom_label_hist(const int32_t* d_idx, int32_t idx_stride, const int32_t* d_labels, int64_t N,
                      int64_t sample_offset, int32_t M, int32_t n_classes, int32_t* d_counts, int64_t* d_first,
                      void* stream);
/* Same with frequency weights, for winners d_idx [N] (stride 1): d_counts float64 [M, n_classes] = sum of the
 * weights per cell, added per winner in ascending sample order (the same on every run for M <= 24576, so a tie
 * between two classes cannot flip between runs), and d_first = smallest global sample index among the samples of
 * the cell with weight > 0 (statistics.mode over the samples that are present).  The samples are grouped by winner
 * in d_workspace (dbgsom_label_hist_weighted_workspace_bytes(N, M) bytes). */
size_t dbgsom_label_hist_weighted_workspace_bytes(int64_t N, int32_t M);
int dbgsom_label_hist_weighted(const int32_t* d_idx, const int32_t* d_labels, const double* d_weight, int64_t N,
                               int64_t sample_offset, int32_t M, int32_t n_classes, double* d_counts, int64_t* d_first,
                               void* d_workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * hop matrix on the device (SURVEY.md section 8(f) rank 2)
 * replaces  nx.floyd_warshall_numpy(self.som_)  dbgsom/BaseSom.py:401 (also :367, :235)
 * d_adj int32 [M, 4]: neighbour indices of every neuron on the 4-connected grid graph, -1 = none.
 * d_hop uint16 [M, ldh]: shortest-path hop counts, 0xFFFF = unreachable.  One BFS per source
 * (unit edges), M <= DBGSOM_HOPS_MAX_M, else DBGSOM_E_UNSUPPORTED (the caller then uses its host BFS).
 */
#define DBGSOM_HOPS_MAX_M 28000
int dbgsom_hops(const int32_t* d_adj, int32_t M, uint16_t* d_hop, int64_t ldh, void* stream);

/* ------------------------------------------------------------------------------------------
 * non-negative sparse coding (SURVEY.md section 8(f) rank 3)
 * replaces  the scikit-learn call of BaseSom.transform  dbgsom/BaseSom.py:241-268
 *           SparseCoder(dictionary=normalize(W), positive_code=True, transform_alpha=0,
 *                       transform_algorithm="lasso_lars").transform(normalize(X))
 *           (also the first step of SomClassifier.predict_proba, dbgsom/SomClassifier.py:178-220)
 * i.e. per sample scikit-learn 1.9's `_lars_path_solver` (Gram mode, method "lasso", positive, alpha_min 0,
 * max_iter 1000), restated in csrc/lars_core.cuh; one CUDA thread per sample.
 *   d_gram [M, M]  = Wn Wn^T  (Wn = row-normalised prototypes), d_cov [N, M] = Xn Wn^T, float64;
 *   n_features = D (scales alpha like the reference); cholesky_capacity = largest active set the scratch is
 *   sized for; d_rows = NULL or a list of N sample indices to process (rerun of the flagged ones);
 *   d_code [N(all), M] float64 coefficients; d_status [N(all)] int32: bit 0 = the active set outgrew
 *   cholesky_capacity (rerun with a larger one), bits 1-3 informational (early stop / degenerate regressor /
 *   simultaneous sign changes, all handled as the reference does).
 *   workspace: dbgsom_sparse_code_workspace_bytes(threads, M, cholesky_capacity); the call uses as many threads
 *   (multiples of 128) as the workspace holds, so any size >= 128 threads' worth works.
 */
size_t dbgsom_sparse_code_workspace_bytes(int64_t n_threads, int32_t M, int32_t cholesky_capacity);
int dbgsom_sparse_code(const double* d_gram, const double* d_cov, int64_t N, int32_t M, int32_t n_features,
                       int32_t max_iter, int32_t cholesky_capacity, const int32_t* d_rows, double* d_code,
                       int32_t* d_status, void* d_workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DBGSOM_B200_H */
