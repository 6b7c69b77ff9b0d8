// Shared device helpers and internal launcher declarations (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "ge2e_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "ge2e_b200 is written for sm_100a only"
#endif

namespace ge2e {

constexpr float kCosDelta = 1e-8f;  // F.cosine_similarity eps (s3:57, s3:70)
#define GE2E_MAX_PEERS 8             // ranks of one NVSwitch domain served by the peer-memory entry points
constexpr int kWarp = 32;

// thread-local record of the last CUDA failure, exposed through the C ABI
void set_cuda_error(cudaError_t e);
// host-side count of kernel launches issued by this library (bench.py's gpu_launches)
void count_launch(int n = 1);

#define GE2E_CUDA_TRY(expr)                    \
  do {                                         \
    cudaError_t _e = (expr);                   \
    if (_e != cudaSuccess) {                   \
      ::ge2e::set_cuda_error(_e);              \
      return GE2E_ERR_LAUNCH;                  \
    }                                          \
  } while (0)

// after every <<<>>>: count the launch and surface launch-configuration errors
#define GE2E_LAUNCHED()                        \
  do {                                         \
    ::ge2e::count_launch(1);                   \
    GE2E_CUDA_TRY(cudaGetLastError());         \
  } while (0)

// Backward of x -> x_hat = x / max(|x|, delta) as F.cosine_similarity differentiates it: the norm's VALUE is
// clamped but its derivative x / |x| is kept, so
//   dx = (dx_hat - x_hat (x_hat . dx_hat) s) / max(|x|, delta),   s = max(|x|, delta) / |x|
// s = 1 above the clamp (the usual Jacobian), delta / |x| below it, 0 at x = 0 (where x_hat = 0).  Callers
// scale their projection x_hat . dx_hat by s.  Below the clamp n is 0 or a normal float (n^2 would underflow
// first), so the approximate division is safe there and keeps the IEEE division's slow path out of the kernels.
__device__ __forceinline__ float clamp_proj_scale(float n) {
  return n >= kCosDelta ? 1.f : (n > 0.f ? __fdividef(kCosDelta, n) : 0.f);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Programmatic dependent launch: a kernel launched with launch_pdl() may start while its stream
// predecessor is still running.  pdl_trigger() lets the successor's CTAs be scheduled as soon as
// every CTA of this grid has executed it (or exited); pdl_wait() blocks until the predecessor grid
// has completed and its writes are visible.  Both are no-ops without the launch attribute.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ float round_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + __expf(-x)); }

// Closes one softmax row (reference s3:119-121) from the OFF-diagonal running state: mx >= Sd is
// the running maximum over all logits incl. the diagonal one, loff = sum_{k != j} exp(S_k - mx).
//   stat = log(sum_k exp S_k + eps)                      (s3:120)
//   q    = 1 - p_j = (sum_{k != j} exp S_k + eps) / (sum_k exp S_k + eps)
//   per  = stat - Sd = -log(1 - q)                        (s3:121), via log1p when q is small
__device__ __forceinline__ void close_softmax_row(float mx, float loff, float Sd, float eps, float& stat,
                                                  float& q, float& per) {
  if (mx > -80.f) {
    const float em = eps * expf(-mx);
    const float Z = loff + expf(Sd - mx) + em;
    stat = mx + logf(Z);
    q = (loff + em) / Z;
  } else {  // every logit below -80: eps dominates
    const float s = expf(mx);
    const float Z = eps + (loff + expf(Sd - mx)) * s;
    stat = logf(Z);
    q = (eps + loff * s) / Z;
  }
  per = (q < 0.5f) ? -log1pf(-q) : stat - Sd;
}

// Block-wide sum; result valid in thread 0.  `red` needs blockDim.x/32 floats.
__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  float t = 0.f;
  if (wid == 0) {
    t = (lane < (int)(blockDim.x >> 5)) ? red[lane] : 0.f;
    t = warp_sum(t);
  }
  return t;
}

// cudaLaunchKernelEx with the programmatic-stream-serialization attribute (see pdl_wait above)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl,
                              Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- launchers implemented in ge2e_simt.cu ------------------------------------------------
struct RowsArgs {
  const float* e_hat;      // [U_local, D]
  const float* c_hat_all;  // [n_total, D]
  const float* cos_diag;   // [U_local]
  int n_local, n_total, spk_offset, M, D;
  const float* w;
  const float* b;
  float eps;
  int variant;
};

// row_index (nullable): logical row r = [speaker][utterance] lives at physical row row_index[r] of E / dE
// e_dt / de_dt: ge2e_dtype of E / dE (checked by the C ABI: dE is fp32 or E's type)
// prec: 0 = fp32 operands as they are, 1 = rounded to TF32, 3 = the hi plane of 2 alone, 2 = two fp16 planes [rows][2][D] (hi, lo) in the
// same allocation (D = 128 / 256 / 512 only)
int simt_prep(const void* E, int e_dt, const int32_t* row_index, int n_local, int M, int D, int prec, float* e_hat,
              float* c_hat_local, float* cos_diag, float* accum, cudaStream_t st);
int simt_fwd_rows(const RowsArgs& a, float* row_stat, int32_t* row_kstar, float* row_aux,
                  float* loss_accum, float* per_row_out, float* sim_out, cudaStream_t st);
// grad_rows (nullable): the upstream gradient per local utterance row, in place of the scalar grad_out -- selects the
// row-gradient (RG) instantiations of the backward kernels
int simt_bwd_rows(const RowsArgs& a, const float* row_stat, const int32_t* row_kstar,
                  const float* row_aux, const float* grad_out, const float* grad_rows, float* dE_hat,
                  float* dC_hat_partial, float* dwdb_accum, cudaStream_t st);
// largest M whose backward finalize runs at width D (0: D unsupported); see ge2e_b200_max_utterances
int finalize_max_rows(int D);
int simt_bwd_finalize(const void* E, int e_dt, const int32_t* row_index, const float* dE_hat, const float* dC_hat_local,
                      const float* cos_diag, const float* row_stat, const float* row_aux,
                      const float* row_scale /* nullable: dE_hat row r is g * row_scale[r] * dE_hat[r] */,
                      int n_local, int M, int D,
                      const float* w, const float* b, float eps, int variant,
                      const float* grad_out, const float* grad_rows /* nullable, as in simt_bwd_rows */, void* dE,
                      int de_dt, bool pdl, cudaStream_t st);
// fused single-kernel fwd+bwd step for small batches (ge2e_simt.cu)
bool small_step_supported(int N, int M, int D);
bool small_step_preferred(int N, int M, int D, int variant);   // supported AND faster than the pipeline
size_t small_step_workspace_bytes(int N, int M, int D);
// part: the whole step, or its forward half (through the row losses) / backward half (upstream gradient grad_rows
// per logical row; e_hat, c_hat, cos_diag and the row statistics are inputs) -- reduction "none"
enum { kSmallWhole = 0, kSmallFwd = 1, kSmallBwd = 2 };
int simt_small_step(int part, const void* E, int e_dt, const int32_t* row_index, int N, int M, int D, const float* w,
                    const float* b, float eps, int variant, const float* grad_out, const float* grad_rows, float* e_hat,
                    float* c_hat, float* cos_diag, float* row_stat, int32_t* row_kstar, float* row_aux, float* per_row,
                    float* loss_accum, float* dE_hat, float* dC_hat, float* dwdb, void* dE, int de_dt, void* workspace,
                    cudaStream_t st);
// out_dt: ge2e_dtype of out (in is fp32)
int simt_scale_grads(const float* in, void* out, int out_dt, long long n, const float* dwdb_in, float* dwdb_out,
                     const float* g, cudaStream_t st);
int simt_scale_bias_sgd(float* w, float* b, float* dw, float* db, float max_norm, float lr, float* total_norm,
                        bool pdl, cudaStream_t st);
int simt_threshold_counts(const float* sim, int N, int M, const float* thresholds, int T, long long* accept_all,
                          long long* accept_own, void* scratch, cudaStream_t st);
int simt_gather_spans(const float* bank, const long long* src_off, int rows, long long span, bool vec_ok, float* out,
                      cudaStream_t st);
int simt_centroids(const float* E, int N, int M, int D, float* C, cudaStream_t st);
int simt_utterance_centroids(const float* E, int N, int M, int D, float* Uc, cudaStream_t st);
int simt_calc_loss(const float* S, int N, int M, float eps, int variant, float* loss,
                   float* per_row, cudaStream_t st);
int simt_normalize_rows(const float* X, int rows, int D, float* Y, cudaStream_t st);

// ---- launchers implemented in ge2e_tail.cu (model tail: Linear + L2 normalise, tcgen05) -----
bool tail_supported(int U, int H, int D, long long x_row_stride);
int tail_fwd(const float* X, long long x_row_stride, const float* W, const float* bias, int U, int H, int D,
             float* E, float* inv_norm, cudaStream_t st);
int tail_bwd_rows(const float* dE, const float* E, const float* inv_norm, int U, int D, float* dY, float* dbias,
                  cudaStream_t st);
// gradient GEMMs of the Linear layer on tcgen05: dX = dY W (row stride dx_row_stride), dW = dY^T X; either may be null
bool tail_bwd_gemms_supported(int U, int H, int D, long long x_row_stride, long long dx_row_stride);
int tail_bwd_gemms(const float* dY, const float* W, const float* X, long long x_row_stride, int U, int H, int D,
                   float* dX, long long dx_row_stride, float* dW, cudaStream_t st);

// ---- launchers implemented in ge2e_tc.cu (tcgen05 / TMA / TMEM path) ----------------------
bool tc_supported(int n_local, int n_total, int M, int D, int variant);
// fp32-class precision on tensor cores (operands as two fp16 planes, see ge2e_tc.cu): softmax, D = 128 / 256
bool tc_split_supported(int n_local, int n_total, int M, int D, int variant);
// GE2E_TF32 softmax step with MMA1 on fp16 copies of the operands (see PREC_HYB in ge2e_tc.cu); mode: 0 = where it
// was measured faster (default), 1 = every supported shape, -1 = never (tests / A-B timing)
bool tc_hybrid_selected(int n_local, int n_total, int M, int D, int variant);
void tc_set_hybrid(int mode);
void tc_set_trace(unsigned long long* device_buf, int mode);
void tc_set_stamps(unsigned long long* device_buf);
int tc_debug_step_schedule(int u_local, int n_total, int cg, int max_clusters, int* de_begin, int* dc_begin,
                           int* partial, int* units);
int tc_debug_step_model(int u_local, int n_total, int cg, int max_clusters, int* dc_rot, double* finish, double* model);
size_t tc_workspace_bytes(int n_local, int n_total, int M, int D, int variant);
// Buffers of one tc_rows call; a field the call does not use stays null.
struct TcRowsBufs {
  const float* grad_out = nullptr;    // scalar upstream gradient (phases with the centroid pass)
  const float* grad_rows = nullptr;   // per local utterance row, in place of grad_out (the centroid pass alone)
  // row statistics: written where the rows are closed in this call, read where an earlier call closed them
  float* row_stat = nullptr;
  int32_t* row_kstar = nullptr;       // contrast
  float* row_aux = nullptr;
  float* row_scale = nullptr;         // factor of the un-normalised dE_hat rows (rows pass)
  float* loss_accum = nullptr;
  float* per_row = nullptr;           // nullable: [U_local] row losses
  float* dE_hat = nullptr;
  float* dC_hat_partial = nullptr;
  float* dwdb = nullptr;
  // speaker-sharded over peer memory (HOST array of n_ranks device pointers): pass 2 adds its accumulators straight
  // into the owner rank's dC_local[n_total / n_ranks, D] (see ge2e_b200_step_rows_peers)
  float* const* dC_owner = nullptr;
  int n_ranks = 0;
};
// The rows kernels on tensor cores.  prec: 0 TF32, 1 split fp16 planes, 2 one fp16 plane.
// phases = 0: the forward kernel alone (loss and row statistics, either variant).  Otherwise the softmax step:
// 1 = rows pass (loss, row statistics, un-normalised dE_hat + row_scale), 2 = centroid pass (dC_hat_partial,
// {dw, db}) from the row statistics of an earlier rows pass, 3 = both in one launch.  On fp16 planes the forward
// kernel closes the rows before a step that has the rows pass; on TF32 the step closes them itself.
int tc_rows(const RowsArgs& a, int prec, int phases, const TcRowsBufs& b, void* ws, size_t ws_bytes,
            cudaStream_t st);
int simt_peer_publish(const float* src, float* const* dst, int n_dst, bool multicast, long long n_floats, float* zero,
                      long long zero_floats, cudaStream_t st);

}  // namespace ge2e
