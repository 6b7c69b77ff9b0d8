// C ABI of the B200-native GE2E loss: argument checking and path selection only.
// See include/ge2e_b200.h for the contract and the reference lines each entry point replaces.
#include <stdlib.h>

#include <atomic>

#include "ge2e_common.cuh"

namespace ge2e {
static thread_local cudaError_t g_last_cuda_error = cudaSuccess;
void set_cuda_error(cudaError_t e) { g_last_cuda_error = e; }
static std::atomic<unsigned long long> g_launches{0};
void count_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }
}  // namespace ge2e

using namespace ge2e;

namespace {

int check_shape(int n_local, int n_total, int spk_offset, int M, int D) {
  if (n_local <= 0 || n_total <= 0 || M < 2 || D <= 0) return GE2E_ERR_SHAPE;
  if (spk_offset < 0 || spk_offset + n_local > n_total) return GE2E_ERR_SHAPE;
  if ((long long)n_local * M > 0x7fffffffLL / 2) return GE2E_ERR_SHAPE;
  if (D > 1024) return GE2E_ERR_UNSUPPORTED;
  return GE2E_OK;
}

int check_enum(int variant, int precision) {
  if (variant != GE2E_SOFTMAX && variant != GE2E_CONTRAST) return GE2E_ERR_ARGUMENT;
  if (precision != GE2E_FP32 && precision != GE2E_TF32 && precision != GE2E_FP32_SPLIT && precision != GE2E_F16)
    return GE2E_ERR_ARGUMENT;
  return GE2E_OK;
}

// (shape, variant, precision) runs on the tensor-core kernels.  GE2E_TF32 is a permission (uncovered shapes run
// on the SIMT kernels, same operand layout); GE2E_FP32_SPLIT is a demand, because its operand layout (two fp16
// planes) is only understood by the tensor-core kernels: callers check ge2e_b200_path() first.
// fp16 operand planes (a demand, see above): GE2E_FP32_SPLIT (two planes, fp32-class) and GE2E_F16 (one plane)
bool is_planes(int precision) { return precision == GE2E_FP32_SPLIT || precision == GE2E_F16; }
// operand precision code of the tensor-core launchers (ge2e_common.cuh): 0 TF32, 1 split planes, 2 one plane
int tc_prec(int precision) { return precision == GE2E_FP32_SPLIT ? 1 : (precision == GE2E_F16 ? 2 : 0); }

// E is fp32 / bf16 / fp16; dE is fp32 or E's own type
int check_dtypes(int e_dtype, int de_dtype) {
  if (e_dtype != GE2E_DT_F32 && e_dtype != GE2E_DT_BF16 && e_dtype != GE2E_DT_F16) return GE2E_ERR_ARGUMENT;
  if (de_dtype != GE2E_DT_F32 && de_dtype != e_dtype) return GE2E_ERR_ARGUMENT;
  return GE2E_OK;
}

bool on_tc(int n_local, int n_total, int M, int D, int variant, int precision) {
  if (n_local <= 0 || n_total <= 0 || M < 2 || D <= 0) return false;
  if (precision == GE2E_TF32) return tc_supported(n_local, n_total, M, D, variant);
  if (is_planes(precision)) return tc_split_supported(n_local, n_total, M, D, variant);
  return false;
}

}  // namespace

extern "C" {

int ge2e_b200_version(void) { return 102; }

const char* ge2e_b200_strerror(int status) {
  switch (status) {
    case GE2E_OK: return "ok";
    case GE2E_ERR_SHAPE: return "bad shape: need n_local,n_total,D > 0, M >= 2, shard inside [0,n_total)";
    case GE2E_ERR_UNSUPPORTED: return "shape not supported by the requested precision path";
    case GE2E_ERR_ARGUMENT: return "null pointer or unknown variant/precision/dtype";
    case GE2E_ERR_WORKSPACE: return "workspace smaller than ge2e_b200_workspace_bytes()";
    case GE2E_ERR_DEVICE: return "current CUDA device is not compute capability 10.x (sm_100a build)";
    case GE2E_ERR_LAUNCH: return "CUDA launch or driver error (see ge2e_b200_last_cuda_error)";
    default: return "unknown ge2e status";
  }
}

int ge2e_b200_last_cuda_error(void) { return (int)g_last_cuda_error; }

unsigned long long ge2e_b200_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

void ge2e_b200_debug_trace(unsigned long long* device_buf, int kernel) { tc_set_trace(device_buf, kernel); }

void ge2e_b200_debug_stamps(unsigned long long* device_buf) { tc_set_stamps(device_buf); }

void ge2e_b200_debug_hybrid(int mode) { tc_set_hybrid(mode); }

int ge2e_b200_debug_step_schedule(int u_local, int n_total, int cta_group, int max_clusters, int* de_begin_host,
                                  int* dc_begin_host, int* partial_host, int* units_host) {
  if (!de_begin_host || !dc_begin_host || !partial_host || !units_host) return GE2E_ERR_ARGUMENT;
  return tc_debug_step_schedule(u_local, n_total, cta_group, max_clusters, de_begin_host, dc_begin_host,
                                partial_host, units_host);
}

int ge2e_b200_debug_step_model(int u_local, int n_total, int cta_group, int max_clusters, int* dc_rot_host,
                               double* finish_host, double* model_host) {
  if (!dc_rot_host || !finish_host || !model_host) return GE2E_ERR_ARGUMENT;
  return tc_debug_step_model(u_local, n_total, cta_group, max_clusters, dc_rot_host, finish_host, model_host);
}

int ge2e_b200_path(int n_local, int n_total, int M, int D, int variant, int precision) {
  if (check_enum(variant, precision) != GE2E_OK) return GE2E_ERR_ARGUMENT;
  if (is_planes(precision)) return on_tc(n_local, n_total, M, D, variant, precision) ? precision : GE2E_ERR_UNSUPPORTED;
  return on_tc(n_local, n_total, M, D, variant, precision) ? 1 : 0;
}

int ge2e_b200_max_utterances(int D) { return finalize_max_rows(D); }

int ge2e_b200_check_device(void) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return GE2E_ERR_DEVICE;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess)
    return GE2E_ERR_DEVICE;
  return major == 10 ? GE2E_OK : GE2E_ERR_DEVICE;
}

size_t ge2e_b200_workspace_bytes(int n_local, int n_total, int M, int D, int variant, int precision) {
  if (on_tc(n_local, n_total, M, D, variant, precision)) return tc_workspace_bytes(n_local, n_total, M, D, variant);
  return 0;
}

int ge2e_b200_prep_typed(const void* E, int e_dtype, const int32_t* row_index, int n_local, int M, int D,
                         int precision, float* e_hat, float* c_hat_local, float* cos_diag, float* accum,
                         ge2e_stream_t stream) {
  if (!E || !e_hat || !c_hat_local || !cos_diag) return GE2E_ERR_ARGUMENT;
  int rc = check_shape(n_local, n_local, 0, M, D);
  if (rc != GE2E_OK) return rc;
  if ((rc = check_enum(GE2E_SOFTMAX, precision)) != GE2E_OK) return rc;
  if ((rc = check_dtypes(e_dtype, GE2E_DT_F32)) != GE2E_OK) return rc;
  return simt_prep(E, e_dtype, row_index, n_local, M, D, precision, e_hat, c_hat_local, cos_diag, accum,
                   (cudaStream_t)stream);
}

int ge2e_b200_prep_indexed(const float* E, const int32_t* row_index, int n_local, int M, int D, int precision,
                           float* e_hat, float* c_hat_local, float* cos_diag, float* accum,
                           ge2e_stream_t stream) {
  return ge2e_b200_prep_typed(E, GE2E_DT_F32, row_index, n_local, M, D, precision, e_hat, c_hat_local, cos_diag, accum,
                              stream);
}

int ge2e_b200_prep(const float* E, int n_local, int M, int D, int precision, float* e_hat,
                   float* c_hat_local, float* cos_diag, float* accum, ge2e_stream_t stream) {
  return ge2e_b200_prep_typed(E, GE2E_DT_F32, nullptr, n_local, M, D, precision, e_hat, c_hat_local, cos_diag, accum,
                              stream);
}

static int fwd_rows_impl(const float* e_hat, const float* c_hat_all, const float* cos_diag,
                       int n_local, int n_total, int spk_offset, int M, int D, const float* w,
                       const float* b, float eps, int variant, int precision, float* row_stat,
                       int32_t* row_kstar, float* row_aux, float* loss_accum, float* per_row_out,
                       float* sim_out, float* dE_hat, float* row_scale, void* workspace, size_t workspace_bytes,
                       ge2e_stream_t stream) {
  if (!e_hat || !c_hat_all || !cos_diag || !w || !b || !row_stat || !loss_accum)
    return GE2E_ERR_ARGUMENT;
  int rc = check_shape(n_local, n_total, spk_offset, M, D);
  if (rc != GE2E_OK) return rc;
  if ((rc = check_enum(variant, precision)) != GE2E_OK) return rc;
  if (variant == GE2E_CONTRAST && !row_kstar) return GE2E_ERR_ARGUMENT;
  if (variant == GE2E_SOFTMAX && !row_aux) return GE2E_ERR_ARGUMENT;
  RowsArgs a{e_hat, c_hat_all, cos_diag, n_local, n_total, spk_offset, M, D, w, b, eps, variant};
  if (is_planes(precision) && !on_tc(n_local, n_total, M, D, variant, precision)) return GE2E_ERR_UNSUPPORTED;
  if (on_tc(n_local, n_total, M, D, variant, precision)) {
    // the tensor-core path never materialises S: sim_out is an fp32-path feature
    if (sim_out != nullptr) return GE2E_ERR_UNSUPPORTED;
    TcRowsBufs t;
    t.row_stat = row_stat; t.row_kstar = row_kstar; t.row_aux = row_aux; t.loss_accum = loss_accum;
    t.per_row = per_row_out; t.dE_hat = dE_hat; t.row_scale = row_scale;
    // softmax with a backward to follow: the rows pass of the step kernel also leaves the un-normalised dE_hat
    const int phases = (variant == GE2E_SOFTMAX && dE_hat != nullptr && row_scale != nullptr) ? 1 : 0;
    return tc_rows(a, tc_prec(precision), phases, t, workspace, workspace_bytes, (cudaStream_t)stream);
  }
  return simt_fwd_rows(a, row_stat, row_kstar, row_aux, loss_accum, per_row_out, sim_out,
                       (cudaStream_t)stream);
}

int ge2e_b200_fwd_rows(const float* e_hat, const float* c_hat_all, const float* cos_diag,
                       int n_local, int n_total, int spk_offset, int M, int D, const float* w,
                       const float* b, float eps, int variant, int precision, float* row_stat,
                       int32_t* row_kstar, float* row_aux, float* loss_accum, float* per_row_out,
                       float* sim_out, float* dE_hat, float* row_scale, void* workspace, size_t workspace_bytes,
                       ge2e_stream_t stream) {
  return fwd_rows_impl(e_hat, c_hat_all, cos_diag, n_local, n_total, spk_offset, M, D, w, b, eps, variant,
                       precision, row_stat, row_kstar, row_aux, loss_accum, per_row_out, sim_out, dE_hat, row_scale,
                       workspace, workspace_bytes, stream);
}

// grad_rows (nullable): the upstream gradient per local utterance row, in place of the scalar grad_out
static int bwd_rows_impl(const float* e_hat, const float* c_hat_all, const float* cos_diag, const float* row_stat,
                         const int32_t* row_kstar, const float* row_aux, const float* row_scale, int n_local,
                         int n_total, int spk_offset, int M, int D, const float* w, const float* b, float eps,
                         int variant, int precision, const float* grad_out, const float* grad_rows, float* dE_hat,
                         float* dC_hat_partial, float* dwdb_accum, void* workspace, size_t workspace_bytes,
                         ge2e_stream_t stream) {
  if (!e_hat || !c_hat_all || !cos_diag || !row_stat || !w || !b || (!grad_out && !grad_rows) || !dE_hat ||
      !dC_hat_partial || !dwdb_accum)
    return GE2E_ERR_ARGUMENT;
  int rc = check_shape(n_local, n_total, spk_offset, M, D);
  if (rc != GE2E_OK) return rc;
  if ((rc = check_enum(variant, precision)) != GE2E_OK) return rc;
  if (variant == GE2E_CONTRAST && !row_kstar) return GE2E_ERR_ARGUMENT;
  if (variant == GE2E_SOFTMAX && !row_aux) return GE2E_ERR_ARGUMENT;
  RowsArgs a{e_hat, c_hat_all, cos_diag, n_local, n_total, spk_offset, M, D, w, b, eps, variant};
  // the contrast gradient is a 2-nonzeros-per-row gather/scatter: no contraction to put on
  // tensor cores, so both precisions share the SIMT kernel.  Softmax on tensor cores: the forward's rows
  // pass already left the un-normalised dE_hat (row_scale says so); only the centroid pass remains.
  if (is_planes(precision) && (!on_tc(n_local, n_total, M, D, variant, precision) || row_scale == nullptr))
    return GE2E_ERR_UNSUPPORTED;
  if (variant == GE2E_SOFTMAX && row_scale != nullptr && on_tc(n_local, n_total, M, D, variant, precision)) {
    TcRowsBufs t;
    t.grad_out = grad_out; t.grad_rows = grad_rows;
    t.row_stat = const_cast<float*>(row_stat); t.row_aux = const_cast<float*>(row_aux);   // read by the centroid pass
    t.dE_hat = dE_hat; t.dC_hat_partial = dC_hat_partial; t.dwdb = dwdb_accum;
    return tc_rows(a, tc_prec(precision), 2, t, workspace, workspace_bytes, (cudaStream_t)stream);
  }
  return simt_bwd_rows(a, row_stat, row_kstar, row_aux, grad_out, grad_rows, dE_hat, dC_hat_partial, dwdb_accum,
                       (cudaStream_t)stream);
}

int ge2e_b200_bwd_rows(const float* e_hat, const float* c_hat_all, const float* cos_diag,
                       const float* row_stat, const int32_t* row_kstar, const float* row_aux,
                       const float* row_scale, int n_local, int n_total, int spk_offset, int M, int D,
                       const float* w, const float* b, float eps,
                       int variant, int precision, const float* grad_out, float* dE_hat,
                       float* dC_hat_partial, float* dwdb_accum, void* workspace,
                       size_t workspace_bytes, ge2e_stream_t stream) {
  return bwd_rows_impl(e_hat, c_hat_all, cos_diag, row_stat, row_kstar, row_aux, row_scale, n_local, n_total,
                       spk_offset, M, D, w, b, eps, variant, precision, grad_out, nullptr, dE_hat, dC_hat_partial,
                       dwdb_accum, workspace, workspace_bytes, stream);
}

int ge2e_b200_bwd_rows_per_row(const float* e_hat, const float* c_hat_all, const float* cos_diag,
                               const float* row_stat, const int32_t* row_kstar, const float* row_aux,
                               const float* row_scale, int n_local, int n_total, int spk_offset, int M, int D,
                               const float* w, const float* b, float eps, int variant, int precision,
                               const float* grad_rows, float* dE_hat, float* dC_hat_partial, float* dwdb_accum,
                               void* workspace, size_t workspace_bytes, ge2e_stream_t stream) {
  if (!grad_rows) return GE2E_ERR_ARGUMENT;
  return bwd_rows_impl(e_hat, c_hat_all, cos_diag, row_stat, row_kstar, row_aux, row_scale, n_local, n_total,
                       spk_offset, M, D, w, b, eps, variant, precision, nullptr, grad_rows, dE_hat, dC_hat_partial,
                       dwdb_accum, workspace, workspace_bytes, stream);
}

// grad_rows (nullable): as in bwd_rows_impl, per logical utterance row
static int bwd_finalize_impl(const void* E, int e_dtype, const int32_t* row_index, const float* dE_hat,
                             const float* dC_hat_local, const float* cos_diag, const float* row_stat,
                             const float* row_aux, const float* row_scale, int n_local, int M, int D, const float* w,
                             const float* b, float eps, int variant, const float* grad_out, const float* grad_rows,
                             void* dE, int de_dtype, ge2e_stream_t stream) {
  if (!E || !dE_hat || !dC_hat_local || !cos_diag || !row_stat || !w || !b || (!grad_out && !grad_rows) || !dE)
    return GE2E_ERR_ARGUMENT;
  if (variant == GE2E_SOFTMAX && !row_aux) return GE2E_ERR_ARGUMENT;
  int rc = check_shape(n_local, n_local, 0, M, D);
  if (rc != GE2E_OK) return rc;
  if ((rc = check_enum(variant, GE2E_FP32)) != GE2E_OK) return rc;
  if ((rc = check_dtypes(e_dtype, de_dtype)) != GE2E_OK) return rc;
  return simt_bwd_finalize(E, e_dtype, row_index, dE_hat, dC_hat_local, cos_diag, row_stat, row_aux, row_scale, n_local,
                           M, D, w, b, eps, variant, grad_out, grad_rows, dE, de_dtype, true, (cudaStream_t)stream);
}

int ge2e_b200_bwd_finalize_typed(const void* E, int e_dtype, const int32_t* row_index, const float* dE_hat,
                                 const float* dC_hat_local, const float* cos_diag, const float* row_stat,
                                 const float* row_aux, const float* row_scale, int n_local, int M, int D,
                                 const float* w, const float* b, float eps, int variant, const float* grad_out,
                                 void* dE, int de_dtype, ge2e_stream_t stream) {
  return bwd_finalize_impl(E, e_dtype, row_index, dE_hat, dC_hat_local, cos_diag, row_stat, row_aux, row_scale, n_local,
                           M, D, w, b, eps, variant, grad_out, nullptr, dE, de_dtype, stream);
}

int ge2e_b200_bwd_finalize_per_row_typed(const void* E, int e_dtype, const int32_t* row_index, const float* dE_hat,
                                         const float* dC_hat_local, const float* cos_diag, const float* row_stat,
                                         const float* row_aux, const float* row_scale, int n_local, int M, int D,
                                         const float* w, const float* b, float eps, int variant,
                                         const float* grad_rows, void* dE, int de_dtype, ge2e_stream_t stream) {
  if (!grad_rows) return GE2E_ERR_ARGUMENT;
  return bwd_finalize_impl(E, e_dtype, row_index, dE_hat, dC_hat_local, cos_diag, row_stat, row_aux, row_scale, n_local,
                           M, D, w, b, eps, variant, nullptr, grad_rows, dE, de_dtype, stream);
}

int ge2e_b200_bwd_finalize_indexed(const float* E, const int32_t* row_index, const float* dE_hat,
                                   const float* dC_hat_local, const float* cos_diag, const float* row_stat,
                                   const float* row_aux, const float* row_scale, int n_local, int M, int D,
                                   const float* w, const float* b, float eps, int variant, const float* grad_out,
                                   float* dE, ge2e_stream_t stream) {
  return ge2e_b200_bwd_finalize_typed(E, GE2E_DT_F32, row_index, dE_hat, dC_hat_local, cos_diag, row_stat, row_aux,
                                      row_scale, n_local, M, D, w, b, eps, variant, grad_out, dE, GE2E_DT_F32, stream);
}

int ge2e_b200_bwd_finalize(const float* E, const float* dE_hat, const float* dC_hat_local,
                           const float* cos_diag, const float* row_stat, const float* row_aux,
                           const float* row_scale, int n_local, int M, int D, const float* w, const float* b,
                           float eps, int variant, const float* grad_out, float* dE, ge2e_stream_t stream) {
  return ge2e_b200_bwd_finalize_typed(E, GE2E_DT_F32, nullptr, dE_hat, dC_hat_local, cos_diag, row_stat, row_aux,
                                      row_scale, n_local, M, D, w, b, eps, variant, grad_out, dE, GE2E_DT_F32, stream);
}

int ge2e_b200_gather_spans(const float* bank, const long long* src_off, int rows, long long span, int offsets_aligned,
                           float* out, ge2e_stream_t stream) {
  if (rows < 1 || span < 1) return GE2E_ERR_SHAPE;
  if (!bank || !src_off || !out) return GE2E_ERR_ARGUMENT;
  const bool vec = offsets_aligned != 0 && span % 4 == 0 &&
                   ((reinterpret_cast<uintptr_t>(bank) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  return simt_gather_spans(bank, src_off, rows, span, vec, out, (cudaStream_t)stream);
}

int ge2e_b200_embed_tail_fwd(const float* X, long long x_row_stride, const float* W, const float* bias, int U,
                             int H, int D, float* E, float* inv_norm, ge2e_stream_t stream) {
  if (U < 1 || H < 1 || D < 1) return GE2E_ERR_SHAPE;
  if (!X || !W || !E) return GE2E_ERR_ARGUMENT;
  return tail_fwd(X, x_row_stride, W, bias, U, H, D, E, inv_norm, (cudaStream_t)stream);
}

int ge2e_b200_embed_tail_bwd_rows(const float* dE, const float* E, const float* inv_norm, int U, int D, float* dY,
                                  float* dbias, ge2e_stream_t stream) {
  if (U < 1 || D < 1) return GE2E_ERR_SHAPE;
  if (!dE || !E || !inv_norm || !dY) return GE2E_ERR_ARGUMENT;
  return tail_bwd_rows(dE, E, inv_norm, U, D, dY, dbias, (cudaStream_t)stream);
}

int ge2e_b200_embed_tail_bwd_gemms_supported(int U, int H, int D, long long x_row_stride, long long dx_row_stride) {
  return tail_bwd_gemms_supported(U, H, D, x_row_stride, dx_row_stride) ? 1 : 0;
}

int ge2e_b200_embed_tail_bwd_gemms(const float* dY, const float* W, const float* X, long long x_row_stride, int U,
                                   int H, int D, float* dX, long long dx_row_stride, float* dW, ge2e_stream_t stream) {
  if (U < 1 || H < 1 || D < 1) return GE2E_ERR_SHAPE;
  if (!dY || (!dX && !dW) || (dX && !W) || (dW && !X)) return GE2E_ERR_ARGUMENT;
  return tail_bwd_gemms(dY, W, X, x_row_stride, U, H, D, dX, dx_row_stride, dW, (cudaStream_t)stream);
}

size_t ge2e_b200_threshold_counts_scratch_bytes(int T) {
  return T < 1 ? 0 : (size_t)(2 * (T + 1) + 1) * sizeof(unsigned long long);
}

int ge2e_b200_threshold_counts(const float* sim, int N, int M, const float* thresholds, int T,
                               long long* accept_all, long long* accept_own, void* scratch,
                               size_t scratch_bytes, ge2e_stream_t stream) {
  if (N < 1 || M < 1) return GE2E_ERR_SHAPE;
  if (!sim || !thresholds || !accept_all || !accept_own || !scratch) return GE2E_ERR_ARGUMENT;
  if (T < 1) return GE2E_ERR_SHAPE;
  if (scratch_bytes < ge2e_b200_threshold_counts_scratch_bytes(T)) return GE2E_ERR_WORKSPACE;
  return simt_threshold_counts(sim, N, M, thresholds, T, accept_all, accept_own, scratch, (cudaStream_t)stream);
}

int ge2e_b200_scale_bias_sgd(float* w, float* b, float* dw, float* db, float max_norm, float lr,
                             float* total_norm, ge2e_stream_t stream) {
  if (!w || !b || !dw || !db) return GE2E_ERR_ARGUMENT;
  if (!(max_norm > 0.f) || !(lr >= 0.f)) return GE2E_ERR_ARGUMENT;
  return simt_scale_bias_sgd(w, b, dw, db, max_norm, lr, total_norm, true, (cudaStream_t)stream);
}

// true when (shape, variant, precision) runs the softmax step on tensor cores: there the forward's rows pass
// leaves an UN-NORMALISED dE_hat plus row_scale, and the backward is the centroid pass alone
static bool tc_softmax_step(int n_local, int n_total, int M, int D, int variant, int precision) {
  return variant == GE2E_SOFTMAX && on_tc(n_local, n_total, M, D, variant, precision);
}

static bool use_small_step(int N, int M, int D, int variant, int precision);

// Per-utterance losses on a shape of the single-kernel step: its two halves (kSmallFwd / kSmallBwd), where the caller's
// workspace has room for them.  A workspace sized by ge2e_b200_workspace_bytes() keeps the staged kernels.
static bool use_small_halves(int N, int M, int D, int variant, int precision, const void* workspace,
                             size_t workspace_bytes) {
  return use_small_step(N, M, D, variant, precision) && workspace != nullptr &&
         workspace_bytes >= small_step_workspace_bytes(N, M, D);
}

// per_row (nullable): [N*M] row losses in logical order
static int forward_impl(const void* E, int e_dtype, const int32_t* row_index, int N, int M, int D, const float* w,
                        const float* b, float eps, int variant, int precision, float* e_hat, float* c_hat,
                        float* cos_diag, float* row_stat, int32_t* row_kstar, float* row_aux, float* accum,
                        float* dE_hat, float* row_scale, float* per_row, void* workspace, size_t workspace_bytes,
                        ge2e_stream_t stream) {
  if (!accum) return GE2E_ERR_ARGUMENT;
  int rc = check_enum(variant, precision);
  if (rc != GE2E_OK) return rc;
  if ((rc = check_dtypes(e_dtype, GE2E_DT_F32)) != GE2E_OK) return rc;
  if (per_row != nullptr && use_small_halves(N, M, D, variant, precision, workspace, workspace_bytes)) {
    if (!E || !w || !b || !e_hat || !c_hat || !cos_diag || !row_stat) return GE2E_ERR_ARGUMENT;
    if ((rc = check_shape(N, N, 0, M, D)) != GE2E_OK) return rc;
    if (variant == GE2E_CONTRAST && !row_kstar) return GE2E_ERR_ARGUMENT;
    if (variant == GE2E_SOFTMAX && !row_aux) return GE2E_ERR_ARGUMENT;
    return simt_small_step(kSmallFwd, E, e_dtype, row_index, N, M, D, w, b, eps, variant, nullptr, nullptr, e_hat, c_hat,
                           cos_diag, row_stat, row_kstar, row_aux, per_row, accum, nullptr, nullptr, nullptr, nullptr,
                           GE2E_DT_F32, workspace, (cudaStream_t)stream);
  }
  // tensor-core path: prep and the rows kernel are adjacent in the stream, the second one is launched
  // programmatically under the first one's tail
  rc = ge2e_b200_prep_typed(E, e_dtype, row_index, N, M, D, precision, e_hat, c_hat, cos_diag, accum, stream);
  if (rc != GE2E_OK) return rc;
  return fwd_rows_impl(e_hat, c_hat, cos_diag, N, N, 0, M, D, w, b, eps, variant, precision, row_stat, row_kstar,
                       row_aux, accum, per_row, nullptr, dE_hat, row_scale, workspace, workspace_bytes, stream);
}

int ge2e_b200_forward_typed(const void* E, int e_dtype, const int32_t* row_index, int N, int M, int D, const float* w,
                            const float* b, float eps, int variant, int precision, float* e_hat, float* c_hat,
                            float* cos_diag, float* row_stat, int32_t* row_kstar, float* row_aux, float* accum,
                            float* dE_hat, float* row_scale, void* workspace, size_t workspace_bytes,
                            ge2e_stream_t stream) {
  return forward_impl(E, e_dtype, row_index, N, M, D, w, b, eps, variant, precision, e_hat, c_hat, cos_diag, row_stat,
                      row_kstar, row_aux, accum, dE_hat, row_scale, nullptr, workspace, workspace_bytes, stream);
}

int ge2e_b200_forward_per_row_typed(const void* E, int e_dtype, const int32_t* row_index, int N, int M, int D,
                                    const float* w, const float* b, float eps, int variant, int precision, float* e_hat,
                                    float* c_hat, float* cos_diag, float* row_stat, int32_t* row_kstar, float* row_aux,
                                    float* accum, float* dE_hat, float* row_scale, float* per_row, void* workspace,
                                    size_t workspace_bytes, ge2e_stream_t stream) {
  if (!per_row) return GE2E_ERR_ARGUMENT;
  return forward_impl(E, e_dtype, row_index, N, M, D, w, b, eps, variant, precision, e_hat, c_hat, cos_diag, row_stat,
                      row_kstar, row_aux, accum, dE_hat, row_scale, per_row, workspace, workspace_bytes, stream);
}

int ge2e_b200_forward_indexed(const float* E, const int32_t* row_index, int N, int M, int D, const float* w,
                              const float* b, float eps, int variant, int precision, float* e_hat, float* c_hat,
                              float* cos_diag, float* row_stat, int32_t* row_kstar, float* row_aux, float* accum,
                              float* dE_hat, float* row_scale, void* workspace, size_t workspace_bytes,
                              ge2e_stream_t stream) {
  return ge2e_b200_forward_typed(E, GE2E_DT_F32, row_index, N, M, D, w, b, eps, variant, precision, e_hat, c_hat,
                                 cos_diag, row_stat, row_kstar, row_aux, accum, dE_hat, row_scale, workspace,
                                 workspace_bytes, stream);
}

int ge2e_b200_forward(const float* E, int N, int M, int D, const float* w, const float* b, float eps,
                      int variant, int precision, float* e_hat, float* c_hat, float* cos_diag,
                      float* row_stat, int32_t* row_kstar, float* row_aux, float* accum, float* dE_hat,
                      float* row_scale, void* workspace, size_t workspace_bytes, ge2e_stream_t stream) {
  return ge2e_b200_forward_indexed(E, nullptr, N, M, D, w, b, eps, variant, precision, e_hat, c_hat, cos_diag,
                                   row_stat, row_kstar, row_aux, accum, dE_hat, row_scale, workspace, workspace_bytes,
                                   stream);
}

static int backward_impl(const void* E, int e_dtype, const int32_t* row_index, const float* e_hat, const float* c_hat,
                         const float* cos_diag, const float* row_stat, const int32_t* row_kstar, const float* row_aux,
                         const float* row_scale, int N, int M, int D, const float* w, const float* b, float eps,
                         int variant, int precision, const float* grad_out, const float* grad_rows, float* dE_hat,
                         float* dC_hat, float* accum, void* dE, int de_dtype, void* workspace, size_t workspace_bytes,
                         ge2e_stream_t stream) {
  if (!accum) return GE2E_ERR_ARGUMENT;
  if (check_dtypes(e_dtype, de_dtype) != GE2E_OK) return GE2E_ERR_ARGUMENT;
  if (M > finalize_max_rows(D)) return GE2E_ERR_UNSUPPORTED;     // before the rows kernels run
  if (grad_rows != nullptr && use_small_halves(N, M, D, variant, precision, workspace, workspace_bytes)) {
    if (!E || !e_hat || !c_hat || !cos_diag || !row_stat || !w || !b || !dE_hat || !dC_hat || !dE)
      return GE2E_ERR_ARGUMENT;
    int rc = check_shape(N, N, 0, M, D);
    if (rc != GE2E_OK) return rc;
    if ((rc = check_enum(variant, precision)) != GE2E_OK) return rc;
    if (variant == GE2E_CONTRAST && !row_kstar) return GE2E_ERR_ARGUMENT;
    if (variant == GE2E_SOFTMAX && !row_aux) return GE2E_ERR_ARGUMENT;
    return simt_small_step(kSmallBwd, E, e_dtype, row_index, N, M, D, w, b, eps, variant, nullptr, grad_rows,
                           const_cast<float*>(e_hat), const_cast<float*>(c_hat), const_cast<float*>(cos_diag),
                           const_cast<float*>(row_stat), const_cast<int32_t*>(row_kstar), const_cast<float*>(row_aux),
                           nullptr, nullptr, dE_hat, dC_hat, accum + 1, dE, de_dtype, workspace, (cudaStream_t)stream);
  }
  // row_scale is meaningful only where the forward produced it
  const float* scale = tc_softmax_step(N, N, M, D, variant, precision) ? row_scale : nullptr;
  int rc = bwd_rows_impl(e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, scale, N, N, 0, M, D, w, b, eps, variant,
                         precision, grad_out, grad_rows, dE_hat, dC_hat, accum + 1, workspace, workspace_bytes, stream);
  if (rc != GE2E_OK) return rc;
  // the finalize kernel directly follows the dC_hat tensor-core kernel: programmatic launch
  return bwd_finalize_impl(E, e_dtype, row_index, dE_hat, dC_hat, cos_diag, row_stat, row_aux, scale, N, M, D, w, b, eps,
                           variant, grad_out, grad_rows, dE, de_dtype, stream);
}

int ge2e_b200_backward_typed(const void* E, int e_dtype, const int32_t* row_index, const float* e_hat,
                             const float* c_hat, const float* cos_diag, const float* row_stat, const int32_t* row_kstar,
                             const float* row_aux, const float* row_scale, int N, int M, int D, const float* w,
                             const float* b, float eps, int variant, int precision, const float* grad_out,
                             float* dE_hat, float* dC_hat, float* accum, void* dE, int de_dtype, void* workspace,
                             size_t workspace_bytes, ge2e_stream_t stream) {
  return backward_impl(E, e_dtype, row_index, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, row_scale, N, M, D,
                       w, b, eps, variant, precision, grad_out, nullptr, dE_hat, dC_hat, accum, dE, de_dtype, workspace,
                       workspace_bytes, stream);
}

int ge2e_b200_backward_per_row_typed(const void* E, int e_dtype, const int32_t* row_index, const float* e_hat,
                                     const float* c_hat, const float* cos_diag, const float* row_stat,
                                     const int32_t* row_kstar, const float* row_aux, const float* row_scale, int N,
                                     int M, int D, const float* w, const float* b, float eps, int variant,
                                     int precision, const float* grad_rows, float* dE_hat, float* dC_hat, float* accum,
                                     void* dE, int de_dtype, void* workspace, size_t workspace_bytes,
                                     ge2e_stream_t stream) {
  if (!grad_rows) return GE2E_ERR_ARGUMENT;
  return backward_impl(E, e_dtype, row_index, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, row_scale, N, M, D,
                       w, b, eps, variant, precision, nullptr, grad_rows, dE_hat, dC_hat, accum, dE, de_dtype,
                       workspace, workspace_bytes, stream);
}

int ge2e_b200_backward_indexed(const float* E, const int32_t* row_index, const float* e_hat, const float* c_hat,
                               const float* cos_diag, const float* row_stat, const int32_t* row_kstar,
                               const float* row_aux, const float* row_scale, int N, int M, int D, const float* w,
                               const float* b, float eps, int variant, int precision, const float* grad_out,
                               float* dE_hat, float* dC_hat, float* accum, float* dE, void* workspace,
                               size_t workspace_bytes, ge2e_stream_t stream) {
  return ge2e_b200_backward_typed(E, GE2E_DT_F32, row_index, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux,
                                  row_scale, N, M, D, w, b, eps, variant, precision, grad_out, dE_hat, dC_hat, accum, dE,
                                  GE2E_DT_F32, workspace, workspace_bytes, stream);
}

int ge2e_b200_backward(const float* E, const float* e_hat, const float* c_hat, const float* cos_diag,
                       const float* row_stat, const int32_t* row_kstar, const float* row_aux, const float* row_scale,
                       int N, int M, int D, const float* w, const float* b, float eps, int variant, int precision,
                       const float* grad_out, float* dE_hat, float* dC_hat, float* accum, float* dE,
                       void* workspace, size_t workspace_bytes, ge2e_stream_t stream) {
  return ge2e_b200_backward_indexed(E, nullptr, e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, row_scale, N, M,
                                    D, w, b, eps, variant, precision, grad_out, dE_hat, dC_hat, accum, dE, workspace,
                                    workspace_bytes, stream);
}

// ---- forward rows + backward rows in one call (what a captured step issues) -----------------
int ge2e_b200_step_rows(const float* e_hat, const float* c_hat_all, const float* cos_diag, int n_local, int n_total,
                        int spk_offset, int M, int D, const float* w, const float* b, float eps, int variant,
                        int precision, const float* grad_out, float* row_stat, int32_t* row_kstar, float* row_aux,
                        float* row_scale, float* accum, float* dE_hat, float* dC_hat_partial, void* workspace,
                        size_t workspace_bytes, ge2e_stream_t stream) {
  if (!e_hat || !c_hat_all || !cos_diag || !w || !b || !grad_out || !row_stat || !row_aux || !row_scale || !accum ||
      !dE_hat || !dC_hat_partial)
    return GE2E_ERR_ARGUMENT;
  int rc = check_shape(n_local, n_total, spk_offset, M, D);
  if (rc != GE2E_OK) return rc;
  if ((rc = check_enum(variant, precision)) != GE2E_OK) return rc;
  if (variant == GE2E_CONTRAST && !row_kstar) return GE2E_ERR_ARGUMENT;
  if (tc_softmax_step(n_local, n_total, M, D, variant, precision)) {
    // both passes of the step kernel, in which pass 2 waits per utterance tile for the row sums of pass 1
    // ({loss, dw, db} += into accum: zeroed by prep)
    RowsArgs a{e_hat, c_hat_all, cos_diag, n_local, n_total, spk_offset, M, D, w, b, eps, variant};
    TcRowsBufs t;
    t.grad_out = grad_out; t.row_stat = row_stat; t.row_kstar = row_kstar; t.row_aux = row_aux; t.row_scale = row_scale;
    t.loss_accum = accum; t.dE_hat = dE_hat; t.dC_hat_partial = dC_hat_partial; t.dwdb = accum + 1;
    return tc_rows(a, tc_prec(precision), 3, t, workspace, workspace_bytes, (cudaStream_t)stream);
  }
  if (is_planes(precision)) return GE2E_ERR_UNSUPPORTED;
  rc = fwd_rows_impl(e_hat, c_hat_all, cos_diag, n_local, n_total, spk_offset, M, D, w, b, eps, variant, precision,
                     row_stat, row_kstar, row_aux, accum, nullptr, nullptr, nullptr, nullptr, workspace, workspace_bytes,
                     stream);
  if (rc != GE2E_OK) return rc;
  return ge2e_b200_bwd_rows(e_hat, c_hat_all, cos_diag, row_stat, row_kstar, row_aux, nullptr, n_local, n_total,
                            spk_offset, M, D, w, b, eps, variant, precision, grad_out, dE_hat, dC_hat_partial, accum + 1,
                            workspace, workspace_bytes, stream);
}

// ---- speaker-sharded step over peer memory (one NVSwitch domain) ---------------------------
int ge2e_b200_peer_publish(const float* src, float* const* dst_host, int n_dst, int multicast, long long n_floats,
                           float* zero, long long zero_floats, ge2e_stream_t stream) {
  if (!src || !dst_host) return GE2E_ERR_ARGUMENT;
  if (n_dst < 1 || n_dst > GE2E_MAX_PEERS || n_floats < 0 || n_floats % 4 != 0 || zero_floats < 0 || zero_floats % 4 != 0 ||
      (multicast && n_dst != 1))
    return GE2E_ERR_SHAPE;
  for (int r = 0; r < n_dst; ++r)
    if (!dst_host[r] || (reinterpret_cast<uintptr_t>(dst_host[r]) & 15) != 0) return GE2E_ERR_ARGUMENT;
  if ((reinterpret_cast<uintptr_t>(src) & 15) != 0 || (zero_floats > 0 && (!zero || (reinterpret_cast<uintptr_t>(zero) & 15) != 0)))
    return GE2E_ERR_ARGUMENT;
  return simt_peer_publish(src, dst_host, n_dst, multicast != 0, n_floats, zero, zero_floats, (cudaStream_t)stream);
}

int ge2e_b200_step_rows_peers(const float* e_hat, const float* c_hat_all, const float* cos_diag, int n_local, int n_total,
                              int spk_offset, int M, int D, const float* w, const float* b, float eps, int variant,
                              int precision, const float* grad_out, float* row_stat, int32_t* row_kstar, float* row_aux,
                              float* row_scale, float* accum, float* dE_hat, float* const* dC_owner_host, int n_ranks,
                              void* workspace, size_t workspace_bytes, ge2e_stream_t stream) {
  if (!e_hat || !c_hat_all || !cos_diag || !w || !b || !grad_out || !row_stat || !row_aux || !row_scale || !accum ||
      !dE_hat || !dC_owner_host)
    return GE2E_ERR_ARGUMENT;
  int rc = check_shape(n_local, n_total, spk_offset, M, D);
  if (rc != GE2E_OK) return rc;
  if ((rc = check_enum(variant, precision)) != GE2E_OK) return rc;
  if (n_ranks < 2 || n_ranks > GE2E_MAX_PEERS || n_local * n_ranks != n_total) return GE2E_ERR_SHAPE;
  // only the tensor-core softmax step flushes through peer memory; everything else keeps the reduce-scatter
  if (!tc_softmax_step(n_local, n_total, M, D, variant, precision)) return GE2E_ERR_UNSUPPORTED;
  RowsArgs a{e_hat, c_hat_all, cos_diag, n_local, n_total, spk_offset, M, D, w, b, eps, variant};
  TcRowsBufs t;
  t.grad_out = grad_out; t.row_stat = row_stat; t.row_kstar = row_kstar; t.row_aux = row_aux; t.row_scale = row_scale;
  t.loss_accum = accum; t.dE_hat = dE_hat; t.dwdb = accum + 1; t.dC_owner = dC_owner_host; t.n_ranks = n_ranks;
  return tc_rows(a, tc_prec(precision), 3, t, workspace, workspace_bytes, (cudaStream_t)stream);
}

int ge2e_b200_bwd_rows_peers_per_row(const float* e_hat, const float* c_hat_all, const float* cos_diag,
                                     const float* row_stat, const float* row_aux, const float* row_scale, int n_local,
                                     int n_total, int spk_offset, int M, int D, const float* w, const float* b,
                                     float eps, int variant, int precision, const float* grad_rows, float* dE_hat,
                                     float* dwdb_accum, float* const* dC_owner_host, int n_ranks, void* workspace,
                                     size_t workspace_bytes, ge2e_stream_t stream) {
  // row_scale: the forward's rows pass prepared dE_hat, so only the centroid pass remains
  if (!e_hat || !c_hat_all || !cos_diag || !row_stat || !row_aux || !row_scale || !w || !b || !grad_rows || !dE_hat ||
      !dwdb_accum || !dC_owner_host)
    return GE2E_ERR_ARGUMENT;
  int rc = check_shape(n_local, n_total, spk_offset, M, D);
  if (rc != GE2E_OK) return rc;
  if ((rc = check_enum(variant, precision)) != GE2E_OK) return rc;
  if (n_ranks < 2 || n_ranks > GE2E_MAX_PEERS || n_local * n_ranks != n_total) return GE2E_ERR_SHAPE;
  if (!tc_softmax_step(n_local, n_total, M, D, variant, precision)) return GE2E_ERR_UNSUPPORTED;
  RowsArgs a{e_hat, c_hat_all, cos_diag, n_local, n_total, spk_offset, M, D, w, b, eps, variant};
  TcRowsBufs t;
  t.grad_rows = grad_rows;
  t.row_stat = const_cast<float*>(row_stat); t.row_aux = const_cast<float*>(row_aux);   // read by the centroid pass
  t.dE_hat = dE_hat; t.dwdb = dwdb_accum; t.dC_owner = dC_owner_host; t.n_ranks = n_ranks;
  return tc_rows(a, tc_prec(precision), 2, t, workspace, workspace_bytes, (cudaStream_t)stream);
}

// grad_rows (nullable): per local utterance row, in place of grad_out
static int contrast_bwd_rows_peers_impl(const float* e_hat, const float* c_hat_all, const float* cos_diag,
                                        const float* row_stat, const int32_t* row_kstar, int n_local, int n_total,
                                        int spk_offset, int M, int D, const float* w, const float* b, float eps,
                                        int precision, const float* grad_out, const float* grad_rows, float* dE_hat,
                                        float* dwdb_accum, float* const* dC_owner_host, int n_ranks,
                                        ge2e_stream_t stream) {
  if (!e_hat || !c_hat_all || !cos_diag || !row_stat || !row_kstar || !w || !b || (!grad_out && !grad_rows) ||
      !dE_hat || !dwdb_accum || !dC_owner_host)
    return GE2E_ERR_ARGUMENT;
  int rc = check_shape(n_local, n_total, spk_offset, M, D);
  if (rc != GE2E_OK) return rc;
  if ((rc = check_enum(GE2E_CONTRAST, precision)) != GE2E_OK) return rc;
  if (n_ranks < 2 || n_ranks > GE2E_MAX_PEERS || n_local * n_ranks != n_total) return GE2E_ERR_SHAPE;
  if (is_planes(precision)) return GE2E_ERR_UNSUPPORTED;     // contrast has no fp16-plane path
  // the vector reductions need every owner row 16-byte aligned wherever D allows them
  const uintptr_t align = D % 4 == 0 ? 15 : 3;
  for (int r = 0; r < n_ranks; ++r)
    if (!dC_owner_host[r] || (reinterpret_cast<uintptr_t>(dC_owner_host[r]) & align) != 0) return GE2E_ERR_ARGUMENT;
  RowsArgs a{e_hat, c_hat_all, cos_diag, n_local, n_total, spk_offset, M, D, w, b, eps, GE2E_CONTRAST};
  return simt_contrast_bwd_rows_peers(a, row_stat, row_kstar, grad_out, grad_rows, dE_hat, dwdb_accum, dC_owner_host,
                                      n_ranks, (cudaStream_t)stream);
}

int ge2e_b200_contrast_bwd_rows_peers(const float* e_hat, const float* c_hat_all, const float* cos_diag,
                                      const float* row_stat, const int32_t* row_kstar, int n_local, int n_total,
                                      int spk_offset, int M, int D, const float* w, const float* b, float eps,
                                      int precision, const float* grad_out, float* dE_hat, float* dwdb_accum,
                                      float* const* dC_owner_host, int n_ranks, ge2e_stream_t stream) {
  if (!grad_out) return GE2E_ERR_ARGUMENT;
  return contrast_bwd_rows_peers_impl(e_hat, c_hat_all, cos_diag, row_stat, row_kstar, n_local, n_total, spk_offset,
                                      M, D, w, b, eps, precision, grad_out, nullptr, dE_hat, dwdb_accum,
                                      dC_owner_host, n_ranks, stream);
}

int ge2e_b200_contrast_bwd_rows_peers_per_row(const float* e_hat, const float* c_hat_all, const float* cos_diag,
                                              const float* row_stat, const int32_t* row_kstar, int n_local,
                                              int n_total, int spk_offset, int M, int D, const float* w,
                                              const float* b, float eps, int precision, const float* grad_rows,
                                              float* dE_hat, float* dwdb_accum, float* const* dC_owner_host,
                                              int n_ranks, ge2e_stream_t stream) {
  if (!grad_rows) return GE2E_ERR_ARGUMENT;
  return contrast_bwd_rows_peers_impl(e_hat, c_hat_all, cos_diag, row_stat, row_kstar, n_local, n_total, spk_offset,
                                      M, D, w, b, eps, precision, nullptr, grad_rows, dE_hat, dwdb_accum,
                                      dC_owner_host, n_ranks, stream);
}

// ---- whole step in one call ---------------------------------------------------------------
// 0 = never (A/B timing), 1 = where it is faster than the pipeline (default), 2 = every supported shape (tests)
static std::atomic<int> g_small_mode{1};
static int small_step_mode() { return g_small_mode.load(std::memory_order_relaxed); }
void ge2e_b200_debug_small_step(int mode) { g_small_mode.store(mode < 0 || mode > 2 ? 1 : mode, std::memory_order_relaxed); }

static bool use_small_step(int N, int M, int D, int variant, int precision) {
  const int mode = small_step_mode();
  if (mode == 0 || !(mode == 2 ? small_step_supported(N, M, D) : small_step_preferred(N, M, D, variant))) return false;
  return !on_tc(N, N, M, D, variant, precision);   // the tensor-core path keeps its shapes
}

size_t ge2e_b200_step_workspace_bytes(int N, int M, int D, int variant, int precision) {
  const size_t base = ge2e_b200_workspace_bytes(N, N, M, D, variant, precision);
  const size_t small = use_small_step(N, M, D, variant, precision) ? small_step_workspace_bytes(N, M, D) : 0;
  return base > small ? base : small;
}

int ge2e_b200_step_launches(int N, int M, int D, int variant, int precision) {
  if (check_enum(variant, precision) != GE2E_OK) return GE2E_ERR_ARGUMENT;
  return use_small_step(N, M, D, variant, precision) ? 1 : 0;
}

int ge2e_b200_forward_backward_typed(const void* E, int e_dtype, const int32_t* row_index, int N, int M, int D,
                                     const float* w, const float* b, float eps, int variant, int precision,
                                     const float* grad_out, float* e_hat, float* c_hat, float* cos_diag,
                                     float* row_stat, int32_t* row_kstar, float* row_aux, float* row_scale,
                                     float* accum, float* dE_hat, float* dC_hat, void* dE, int de_dtype,
                                     void* workspace, size_t workspace_bytes, ge2e_stream_t stream) {
  if (!E || !w || !b || !grad_out || !e_hat || !c_hat || !cos_diag || !row_stat || !row_aux || !row_scale || !accum ||
      !dE_hat || !dC_hat || !dE)
    return GE2E_ERR_ARGUMENT;
  int rc = check_shape(N, N, 0, M, D);
  if (rc != GE2E_OK) return rc;
  if ((rc = check_enum(variant, precision)) != GE2E_OK) return rc;
  if ((rc = check_dtypes(e_dtype, de_dtype)) != GE2E_OK) return rc;
  // refused before any launch: never a forward that ran and a finalize that cannot
  if (M > finalize_max_rows(D)) return GE2E_ERR_UNSUPPORTED;
  if (use_small_step(N, M, D, variant, precision)) {
    if (!workspace || workspace_bytes < small_step_workspace_bytes(N, M, D)) return GE2E_ERR_WORKSPACE;
    if (variant == GE2E_CONTRAST && !row_kstar) return GE2E_ERR_ARGUMENT;
    return simt_small_step(kSmallWhole, E, e_dtype, row_index, N, M, D, w, b, eps, variant, grad_out, nullptr, e_hat,
                           c_hat, cos_diag, row_stat, row_kstar, row_aux, nullptr, accum, dE_hat, dC_hat, accum + 1, dE,
                           de_dtype, workspace, (cudaStream_t)stream);
  }
  // prep (zeroes accum) -> rows: every kernel is launched programmatically under its predecessor's tail
  rc = ge2e_b200_prep_typed(E, e_dtype, row_index, N, M, D, precision, e_hat, c_hat, cos_diag, accum, stream);
  if (rc != GE2E_OK) return rc;
  rc = ge2e_b200_step_rows(e_hat, c_hat, cos_diag, N, N, 0, M, D, w, b, eps, variant, precision, grad_out, row_stat,
                           row_kstar, row_aux, row_scale, accum, dE_hat, dC_hat, workspace, workspace_bytes, stream);
  if (rc != GE2E_OK) return rc;
  const float* scale = tc_softmax_step(N, N, M, D, variant, precision) ? row_scale : nullptr;
  return ge2e_b200_bwd_finalize_typed(E, e_dtype, row_index, dE_hat, dC_hat, cos_diag, row_stat, row_aux, scale, N, M, D,
                                      w, b, eps, variant, grad_out, dE, de_dtype, stream);
}

int ge2e_b200_forward_backward(const float* E, const int32_t* row_index, int N, int M, int D, const float* w,
                               const float* b, float eps, int variant, int precision, const float* grad_out,
                               float* e_hat, float* c_hat, float* cos_diag, float* row_stat, int32_t* row_kstar,
                               float* row_aux, float* row_scale, float* accum, float* dE_hat, float* dC_hat,
                               float* dE, void* workspace, size_t workspace_bytes, ge2e_stream_t stream) {
  return ge2e_b200_forward_backward_typed(E, GE2E_DT_F32, row_index, N, M, D, w, b, eps, variant, precision, grad_out,
                                          e_hat, c_hat, cos_diag, row_stat, row_kstar, row_aux, row_scale, accum, dE_hat,
                                          dC_hat, dE, GE2E_DT_F32, workspace, workspace_bytes, stream);
}

int ge2e_b200_scale_grads_typed(const float* dE_in, void* dE_out, int de_dtype, long long n, const float* dwdb_in,
                                float* dwdb_out, const float* grad_out, ge2e_stream_t stream) {
  if (!dE_in || !dE_out || !dwdb_in || !dwdb_out || !grad_out) return GE2E_ERR_ARGUMENT;
  if (check_dtypes(de_dtype, de_dtype) != GE2E_OK) return GE2E_ERR_ARGUMENT;
  if (n < 1) return GE2E_ERR_SHAPE;
  return simt_scale_grads(dE_in, dE_out, de_dtype, n, dwdb_in, dwdb_out, grad_out, (cudaStream_t)stream);
}

int ge2e_b200_scale_grads(const float* dE_in, float* dE_out, long long n, const float* dwdb_in, float* dwdb_out,
                          const float* grad_out, ge2e_stream_t stream) {
  return ge2e_b200_scale_grads_typed(dE_in, dE_out, GE2E_DT_F32, n, dwdb_in, dwdb_out, grad_out, stream);
}

int ge2e_b200_centroids(const float* E, int N, int M, int D, float* C, ge2e_stream_t stream) {
  if (!E || !C) return GE2E_ERR_ARGUMENT;
  if (N <= 0 || M <= 0 || D <= 0) return GE2E_ERR_SHAPE;
  return simt_centroids(E, N, M, D, C, (cudaStream_t)stream);
}

int ge2e_b200_utterance_centroids(const float* E, int N, int M, int D, float* Uc, ge2e_stream_t stream) {
  if (!E || !Uc) return GE2E_ERR_ARGUMENT;
  if (N <= 0 || M < 2 || D <= 0) return GE2E_ERR_SHAPE;
  return simt_utterance_centroids(E, N, M, D, Uc, (cudaStream_t)stream);
}

int ge2e_b200_normalize_rows(const float* X, int rows, int D, float* Y, ge2e_stream_t stream) {
  if (!X || !Y) return GE2E_ERR_ARGUMENT;
  if (rows <= 0 || D <= 0) return GE2E_ERR_SHAPE;
  return simt_normalize_rows(X, rows, D, Y, (cudaStream_t)stream);
}

int ge2e_b200_calc_loss(const float* S, int N, int M, float eps, int variant, float* loss,
                        float* per_row, ge2e_stream_t stream) {
  if (!S || !loss) return GE2E_ERR_ARGUMENT;
  if (N <= 0 || M <= 0) return GE2E_ERR_SHAPE;
  if (variant != GE2E_SOFTMAX && variant != GE2E_CONTRAST) return GE2E_ERR_ARGUMENT;
  return simt_calc_loss(S, N, M, eps, variant, loss, per_row, (cudaStream_t)stream);
}

}  // extern "C"
