// extern "C" entry points of libdbgsom_b200.so (declared in include/dbgsom_b200.h).
#include "common.cuh"

namespace dbgsom {
int run_colstats(const float*, int64_t, int, int64_t, const float*, const double*, double*, cudaStream_t);
int run_prepare_x16(const float*, int64_t, int, int64_t, const float*, float, const int32_t*, uint16_t*, uint16_t*, int64_t,
                    float*, cudaStream_t);
size_t accumulate_perm_offset(int64_t, int);
bool bmu_select_supported(int64_t N, int64_t ld16, int Mpad, int n_bmu, int granule);
int run_prepare_w(const double*, int, int, const float*, float, float*, uint16_t*, uint16_t*, int64_t, int,
                  const int32_t*, float*, double*, float*, cudaStream_t);
int run_exclude_duplicates(const double*, int, int, const int32_t*, float*, unsigned long long*, cudaStream_t);
int run_tile_bounds(const double*, int, int, const double*, float, const int32_t*, const float*, int, float*, cudaStream_t);
int run_prepare_bias(const float*, int, const float*, uint16_t*, float*, cudaStream_t);
int run_row_ops(double*, int, const int32_t*, int, cudaStream_t);
int run_gather_rows(const float*, int64_t, int, const int64_t*, int, double*, cudaStream_t);
size_t accumulate_workspace_bytes(int64_t, int, int);
int run_accumulate(const dbgsom_accumulate_args&, const double*, double*, cudaStream_t);
size_t label_hist_weighted_workspace_bytes(int64_t, int);
int run_label_counts_weighted(const int32_t*, const int32_t*, const double*, int64_t, int, int, double*, void*, cudaStream_t);
size_t smooth_workspace_bytes(int, int);
int run_smooth(const dbgsom_smooth_args&, cudaStream_t);
int run_node_stats(const int32_t*, int, const double*, int, int64_t, const int32_t*, int, double, const double*, double*,
                   cudaStream_t);
int run_label_hist(const int32_t*, int, const int32_t*, const double*, int64_t, int64_t, int, int, int32_t*, int64_t*,
                   cudaStream_t);
int run_umatrix(const double*, int, int, int64_t, const double*, double*, cudaStream_t);
int run_hops(const int32_t*, int, uint16_t*, int64_t, cudaStream_t);
size_t sparse_code_workspace_bytes(int64_t, int, int);
int run_sparse_code(const double*, const double*, int64_t, int, int, int, int, const int32_t*, double*, int32_t*, void*,
                    size_t, cudaStream_t);
}  // namespace dbgsom

using namespace dbgsom;

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

extern "C" {

int dbgsom_abi_version(void) { return DBGSOM_ABI_VERSION; }

const char* dbgsom_status_string(int status) {
  switch (status) {
    case DBGSOM_OK: return "ok";
    case DBGSOM_E_BADARG: return "dbgsom: bad argument (null pointer, non-positive size or unknown enum)";
    case DBGSOM_E_WORKSPACE: return "dbgsom: workspace too small";
    case DBGSOM_E_UNSUPPORTED: return "dbgsom: shape not supported (D must be a multiple of 4 and <= 4096 after padding; rows 16-byte aligned)";
    case DBGSOM_E_DRIVER: return "dbgsom: cuTensorMapEncodeTiled unavailable or failed";
    case DBGSOM_E_NOT_SM100: return "dbgsom: device is not compute capability 10.x (B200)";
    default: break;
  }
  if (status > 0) return cudaGetErrorString(static_cast<cudaError_t>(status));
  return "dbgsom: unknown status";
}

int dbgsom_check_device(int device) {
  int major = 0;
  DBGSOM_CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  return major == 10 ? DBGSOM_OK : DBGSOM_E_NOT_SM100;
}

int dbgsom_colstats(const float* d_X, int64_t N, int D, int64_t ldx, const float* d_shift_row, double* d_moments,
                    void* stream) {
  if (!d_X || !d_shift_row || !d_moments || N <= 0 || D <= 0 || ldx < D) return DBGSOM_E_BADARG;
  return run_colstats(d_X, N, D, ldx, d_shift_row, nullptr, d_moments, as_stream(stream));
}

int dbgsom_colstats_weighted(const float* d_X, int64_t N, int D, int64_t ldx, const float* d_shift_row,
                             const double* d_weight, double* d_moments, void* stream) {
  if (!d_X || !d_shift_row || !d_moments || N <= 0 || D <= 0 || ldx < D) return DBGSOM_E_BADARG;
  return run_colstats(d_X, N, D, ldx, d_shift_row, d_weight, d_moments, as_stream(stream));
}

int dbgsom_prepare_x16(const float* d_X, int64_t N, int D, int64_t ldx, const float* d_shift, float scale,
                       uint16_t* d_X16_hi, uint16_t* d_X16_lo, int64_t ld16, float* d_xnorm16, void* stream) {
  if (!d_X || !d_shift || !d_X16_hi || !d_xnorm16 || N <= 0 || D <= 0 || ldx < D || ld16 < D) return DBGSOM_E_BADARG;
  if (ld16 % 64 != 0) return DBGSOM_E_UNSUPPORTED;
  return run_prepare_x16(d_X, N, D, ldx, d_shift, scale, nullptr, d_X16_hi, d_X16_lo, ld16, d_xnorm16, as_stream(stream));
}

int dbgsom_prepare_x16_sorted(const float* d_X, int64_t N, int D, int64_t ldx, const float* d_shift, float scale,
                              const int32_t* d_perm, uint16_t* d_X16_hi, uint16_t* d_X16_lo, int64_t ld16,
                              float* d_xnorm16, void* stream) {
  if (!d_X || !d_shift || !d_perm || !d_X16_hi || !d_xnorm16 || N <= 0 || D <= 0 || ldx < D || ld16 < D) return DBGSOM_E_BADARG;
  if (ld16 % 64 != 0 || N > 0x7fffffffLL) return DBGSOM_E_UNSUPPORTED;
  return run_prepare_x16(d_X, N, D, ldx, d_shift, scale, d_perm, d_X16_hi, d_X16_lo, ld16, d_xnorm16, as_stream(stream));
}

int dbgsom_bmu_select_supported(int64_t N, int64_t ld16, int32_t Mpad, int32_t n_bmu, int32_t select_granule) {
  return bmu_select_supported(N, ld16, Mpad, n_bmu, select_granule) ? 1 : 0;
}

int dbgsom_prepare_w(const double* d_W, int M, int D, const float* d_shift, float scale, float* d_W32,
                     uint16_t* d_W16_hi, uint16_t* d_W16_lo, int64_t ld16, int Mpad, const int32_t* d_col_of_proto,
                     float* d_wnorm, double* d_wshift, float* d_wmax, void* stream) {
  if (!d_W || !d_W32 || !d_wmax || M <= 0 || D <= 0) return DBGSOM_E_BADARG;
  if (d_W16_hi && (!d_wnorm || !d_shift || !d_wshift || ld16 < D || Mpad < M)) return DBGSOM_E_BADARG;
  return run_prepare_w(d_W, M, D, d_shift, scale, d_W32, d_W16_hi, d_W16_lo, ld16, Mpad, d_col_of_proto, d_wnorm,
                       d_wshift, d_wmax, as_stream(stream));
}

size_t dbgsom_bmu_workspace_bytes(int64_t N, int32_t n_bmu) {
  (void)n_bmu;
  return BmuWorkspace::bytes(N);
}

static int check_bmu_args(const dbgsom_bmu_args* a) {
  if (!a || !a->d_X || !a->d_W || !a->d_W32 || !a->d_wmax || !a->d_idx || !a->d_workspace) return DBGSOM_E_BADARG;
  if (a->N <= 0 || a->D <= 0 || a->M <= 0 || a->ldx < a->D) return DBGSOM_E_BADARG;
  if (a->n_bmu != 1 && a->n_bmu != 2) return DBGSOM_E_BADARG;
  if (a->n_bmu > a->M) return DBGSOM_E_BADARG;
  if (a->want_dist && !a->d_dist) return DBGSOM_E_BADARG;
  if (a->backend != DBGSOM_BMU_SIMT && a->backend != DBGSOM_BMU_TENSOR) return DBGSOM_E_BADARG;
  if (a->backend == DBGSOM_BMU_TENSOR) {
    if (!a->d_X16_hi || !a->d_W16_hi || !a->d_wnorm || !a->d_xnorm16 || !a->d_proto_of_col) return DBGSOM_E_BADARG;
    if (a->n_pass != 1 && a->n_pass != 3) return DBGSOM_E_BADARG;
    if (a->n_pass == 3 && (!a->d_X16_lo || !a->d_W16_lo)) return DBGSOM_E_BADARG;
    if (a->select != DBGSOM_SELECT_OFF) {
      if (a->select != DBGSOM_SELECT_FLAG && a->select != DBGSOM_SELECT_REFINE) return DBGSOM_E_BADARG;
      if (!a->d_tile_mask || a->n_pass != (a->select == DBGSOM_SELECT_FLAG ? 1 : 3)) return DBGSOM_E_BADARG;
      if (!bmu_select_supported(a->N, a->ld16, a->Mpad, a->n_bmu, a->select_granule)) return DBGSOM_E_UNSUPPORTED;
    }
  } else if (a->select != DBGSOM_SELECT_OFF || a->d_row_perm) {
    return DBGSOM_E_BADARG;
  }
  if (a->D % 4 != 0 || a->ldx % 4 != 0 || !aligned16(a->d_X) || !aligned16(a->d_W32) || !aligned16(a->d_W))
    return DBGSOM_E_UNSUPPORTED;
  if (a->workspace_bytes < BmuWorkspace::bytes(a->N)) return DBGSOM_E_WORKSPACE;
  return DBGSOM_OK;
}

int dbgsom_exclude_duplicates(const double* d_W, int M, int D, const int32_t* d_col_of_proto, float* d_wnorm,
                              uint64_t* d_hash, void* stream) {
  if (!d_W || !d_wnorm || !d_hash || M <= 0 || D <= 0) return DBGSOM_E_BADARG;
  return run_exclude_duplicates(d_W, M, D, d_col_of_proto, d_wnorm, reinterpret_cast<unsigned long long*>(d_hash),
                                as_stream(stream));
}

int dbgsom_tile_bounds(const double* d_W, int M, int D, const double* d_wshift, float scale,
                       const int32_t* d_proto_of_col, const float* d_wnorm, int Mpad, float* d_tile_bound, void* stream) {
  if (!d_W || !d_wshift || !d_wnorm || !d_tile_bound || M <= 0 || D <= 0 || Mpad < M) return DBGSOM_E_BADARG;
  if (Mpad % 128 != 0) return DBGSOM_E_UNSUPPORTED;
  return run_tile_bounds(d_W, M, D, d_wshift, scale, d_proto_of_col, d_wnorm, Mpad, d_tile_bound, as_stream(stream));
}

int dbgsom_prepare_bias(const float* d_wnorm, int Mpad, const float* d_wmax, uint16_t* d_Wb16, float* d_bias_scale,
                        void* stream) {
  if (!d_wnorm || !d_wmax || !d_Wb16 || !d_bias_scale || Mpad <= 0) return DBGSOM_E_BADARG;
  return run_prepare_bias(d_wnorm, Mpad, d_wmax, d_Wb16, d_bias_scale, as_stream(stream));
}

int dbgsom_bmu_candidates(const dbgsom_bmu_args* a, void* stream) {
  const int rc = check_bmu_args(a);
  if (rc != DBGSOM_OK) return rc;
  const BmuWorkspace ws = BmuWorkspace::carve(a->d_workspace, a->N);
  if (a->backend == DBGSOM_BMU_SIMT) return launch_bmu_cand_simt(*a, ws, as_stream(stream));
  return launch_bmu_cand_tensor(*a, ws, as_stream(stream));
}

int dbgsom_bmu_resolve(const dbgsom_bmu_args* a, void* stream) {
  const int rc = check_bmu_args(a);
  if (rc != DBGSOM_OK) return rc;
  return launch_bmu_resolve(*a, BmuWorkspace::carve(a->d_workspace, a->N), as_stream(stream));
}

int dbgsom_bmu(const dbgsom_bmu_args* a, void* stream) {
  const int rc = dbgsom_bmu_candidates(a, stream);
  if (rc != DBGSOM_OK) return rc;
  return dbgsom_bmu_resolve(a, stream);
}

size_t dbgsom_accumulate_workspace_bytes(int64_t N, int32_t M, int32_t D) { return accumulate_workspace_bytes(N, M, D); }
size_t dbgsom_accumulate_perm_offset(int64_t N, int32_t M) { return accumulate_perm_offset(N, M); }

int dbgsom_accumulate(const dbgsom_accumulate_args* a, void* stream) {
  return dbgsom_accumulate_weighted(a, nullptr, nullptr, stream);
}

int dbgsom_accumulate_weighted(const dbgsom_accumulate_args* a, const double* d_weight, double* d_class_hist_w,
                               void* stream) {
  if (!a || !a->d_X || !a->d_bmu || !a->d_W || !a->d_part || !a->d_workspace) return DBGSOM_E_BADARG;
  if (d_weight && a->d_labels && a->n_classes > 0 && !d_class_hist_w) return DBGSOM_E_BADARG;
  if (a->N <= 0 || a->D <= 0 || a->M <= 0 || a->ldx < a->D || !(a->inv_total_variance == a->inv_total_variance))
    return DBGSOM_E_BADARG;
  if (a->N > 0x7fffffffLL) return DBGSOM_E_UNSUPPORTED;  // int32 permutation
  if (a->D % 4 != 0 || a->ldx % 4 != 0 || !aligned16(a->d_X) || !aligned16(a->d_W)) return DBGSOM_E_UNSUPPORTED;
  if (a->workspace_bytes < accumulate_workspace_bytes(a->N, a->M, a->D)) return DBGSOM_E_WORKSPACE;
  return run_accumulate(*a, d_weight, d_class_hist_w, as_stream(stream));
}

size_t dbgsom_smooth_workspace_bytes(int32_t M, int32_t D) { return smooth_workspace_bytes(M, D); }

int dbgsom_smooth(const dbgsom_smooth_args* a, void* stream) {
  if (!a || !a->d_part || !a->d_hop || !a->d_kernel_lut || !a->d_W_in || !a->d_W_out || !a->d_change || !a->d_workspace)
    return DBGSOM_E_BADARG;
  if (a->M <= 0 || a->D <= 0 || a->ldh < a->M || a->lut_len <= 0 || a->d_W_in == a->d_W_out) return DBGSOM_E_BADARG;
  if (a->row_end > a->row_begin && (a->row_begin < 0 || a->row_end > a->M)) return DBGSOM_E_BADARG;
  if (a->workspace_bytes < smooth_workspace_bytes(a->M, a->D)) return DBGSOM_E_WORKSPACE;
  return run_smooth(*a, as_stream(stream));
}

int dbgsom_apply_row_ops(double* d_W, int D, const int32_t* d_ops, int n_ops, void* stream) {
  if (!d_W || D <= 0 || n_ops < 0 || (n_ops > 0 && !d_ops)) return DBGSOM_E_BADARG;
  return run_row_ops(d_W, D, d_ops, n_ops, as_stream(stream));
}

int dbgsom_gather_rows(const float* d_X, int64_t ldx, int D, const int64_t* d_rows, int n_rows, double* d_W,
                       void* stream) {
  if (!d_X || !d_rows || !d_W || D <= 0 || n_rows < 0 || ldx < D) return DBGSOM_E_BADARG;
  return run_gather_rows(d_X, ldx, D, d_rows, n_rows, d_W, as_stream(stream));
}

int dbgsom_node_stats(const int32_t* d_idx, int32_t idx_stride, const double* d_dist, int32_t dist_stride, int64_t N,
                      const int32_t* d_pos, int32_t M, double bandwidth, double* d_out, void* stream) {
  if (!d_idx || !d_dist || !d_pos || !d_out || N <= 0 || M <= 0 || idx_stride < 1 || dist_stride < 1)
    return DBGSOM_E_BADARG;
  if (!(bandwidth > 0.0)) return DBGSOM_E_BADARG;
  return run_node_stats(d_idx, idx_stride, d_dist, dist_stride, N, d_pos, M, bandwidth, nullptr, d_out,
                        as_stream(stream));
}

int dbgsom_node_stats_weighted(const int32_t* d_idx, int32_t idx_stride, const double* d_dist, int32_t dist_stride,
                               int64_t N, const int32_t* d_pos, int32_t M, double bandwidth, const double* d_weight,
                               double* d_out, void* stream) {
  if (!d_idx || !d_dist || !d_pos || !d_out || N <= 0 || M <= 0 || idx_stride < 1 || dist_stride < 1)
    return DBGSOM_E_BADARG;
  if (!(bandwidth > 0.0)) return DBGSOM_E_BADARG;
  return run_node_stats(d_idx, idx_stride, d_dist, dist_stride, N, d_pos, M, bandwidth, d_weight, d_out,
                        as_stream(stream));
}

int dbgsom_umatrix(const double* d_W, int32_t M, int32_t D, int64_t ldw, const double* d_colw, double* d_out,
                   void* stream) {
  if (!d_W || !d_colw || !d_out || M <= 0 || D <= 0 || ldw < D) return DBGSOM_E_BADARG;
  return run_umatrix(d_W, M, D, ldw, d_colw, d_out, as_stream(stream));
}

int dbgsom_label_hist(const int32_t* d_idx, int32_t idx_stride, const int32_t* d_labels, int64_t N,
                      int64_t sample_offset, int32_t M, int32_t n_classes, int32_t* d_counts, int64_t* d_first,
                      void* stream) {
  if (!d_idx || !d_labels || !d_counts || !d_first || N <= 0 || M <= 0 || n_classes <= 0 || idx_stride < 1)
    return DBGSOM_E_BADARG;
  return run_label_hist(d_idx, idx_stride, d_labels, nullptr, N, sample_offset, M, n_classes, d_counts, d_first,
                        as_stream(stream));
}

size_t dbgsom_label_hist_weighted_workspace_bytes(int64_t N, int32_t M) {
  return label_hist_weighted_workspace_bytes(N, M);
}

int dbgsom_label_hist_weighted(const int32_t* d_idx, const int32_t* d_labels, const double* d_weight, int64_t N,
                               int64_t sample_offset, int32_t M, int32_t n_classes, double* d_counts, int64_t* d_first,
                               void* d_workspace, size_t workspace_bytes, void* stream) {
  if (!d_idx || !d_labels || !d_counts || !d_first || !d_workspace || N <= 0 || M <= 0 || n_classes <= 0)
    return DBGSOM_E_BADARG;
  if (N > 0x7fffffffLL) return DBGSOM_E_UNSUPPORTED;  // int32 permutation
  if (workspace_bytes < label_hist_weighted_workspace_bytes(N, M)) return DBGSOM_E_WORKSPACE;
  const int rc = run_label_counts_weighted(d_idx, d_labels, d_weight, N, M, n_classes, d_counts, d_workspace,
                                           as_stream(stream));
  if (rc != DBGSOM_OK) return rc;
  return run_label_hist(d_idx, 1, d_labels, d_weight, N, sample_offset, M, n_classes, nullptr, d_first,
                        as_stream(stream));
}

int dbgsom_hops(const int32_t* d_adj, int32_t M, uint16_t* d_hop, int64_t ldh, void* stream) {
  if (!d_adj || !d_hop || M <= 0 || ldh < M) return DBGSOM_E_BADARG;
  if (!aligned16(d_adj)) return DBGSOM_E_UNSUPPORTED;
  return run_hops(d_adj, M, d_hop, ldh, as_stream(stream));
}

size_t dbgsom_sparse_code_workspace_bytes(int64_t n_threads, int32_t M, int32_t cholesky_capacity) {
  return sparse_code_workspace_bytes(n_threads, M, cholesky_capacity);
}

int dbgsom_sparse_code(const double* d_gram, const double* d_cov, int64_t N, int32_t M, int32_t n_features,
                       int32_t max_iter, int32_t cholesky_capacity, const int32_t* d_rows, double* d_code,
                       int32_t* d_status, void* d_workspace, size_t workspace_bytes, void* stream) {
  if (!d_gram || !d_cov || !d_code || !d_status || !d_workspace) return DBGSOM_E_BADARG;
  if (N <= 0 || M <= 0 || n_features <= 0 || max_iter <= 0 || cholesky_capacity <= 0) return DBGSOM_E_BADARG;
  if (workspace_bytes < sparse_code_workspace_bytes(128, M, cholesky_capacity)) return DBGSOM_E_WORKSPACE;
  return run_sparse_code(d_gram, d_cov, N, M, n_features, max_iter, cholesky_capacity, d_rows, d_code, d_status,
                         d_workspace, workspace_bytes, as_stream(stream));
}

}  // extern "C"
