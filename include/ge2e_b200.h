/*
 * ge2e_b200.h -- C ABI of the B200-native GE2E loss (sm_100a only).
 *
 * This is the drop-in boundary for ONE path of gkv856/speaker_embedding_GE2E_loss:
 * GE2ELoss.forward and its autograd backward
 * (embedding_model_GE2E/s3_loss_function_GE2E.py:19-127, called from
 * s4_train_embed_model.py:103,196,200 and s5_eval_model.py:42-43).  The reference is pure
 * Python and has no FFI of its own; these entry points are what a ctypes binding in
 * s3_loss_function_GE2E.py would call (see INTEGRATION.md).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++/torch types.
 *   - Every pointer is a DEVICE pointer unless its name ends in _host.  The caller owns all
 *     memory; the library never allocates, frees or retains pointers => calls are
 *     CUDA-graph capturable.  All calls are asynchronous on `stream` and never synchronise.
 *   - fp32, row-major, contiguous.  Embeddings E[n_local, M, D]; U_local = n_local * M rows.
 *     The _typed entry points also take E (and write dE) in bf16 / fp16: see ge2e_dtype.
 *   - w, b, grad_out are DEVICE scalars (no host sync to read nn.Parameters).
 *   - Return value: 0 on success, a negative ge2e_status otherwise (ge2e_b200_strerror).
 *   - Speaker sharding: a rank owns speakers [spk_offset, spk_offset + n_local) out of
 *     n_total.  Single GPU: n_local == n_total, spk_offset == 0.
 *   - There is NO CPU implementation behind this ABI.
 */
#ifndef GE2E_B200_H_
#define GE2E_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* ge2e_stream_t; /* cudaStream_t */

enum ge2e_status {
  GE2E_OK = 0,
  GE2E_ERR_SHAPE = -1,       /* M < 2, non-positive dims, offsets out of range            */
  GE2E_ERR_UNSUPPORTED = -2, /* shape not supported by the requested precision path       */
  GE2E_ERR_ARGUMENT = -3,    /* null pointer, unknown variant / precision                 */
  GE2E_ERR_WORKSPACE = -4,   /* workspace smaller than ge2e_b200_workspace_bytes()        */
  GE2E_ERR_DEVICE = -5,      /* current device is not compute capability 10.x             */
  GE2E_ERR_LAUNCH = -6       /* CUDA launch / driver error (see ge2e_b200_last_cuda_error) */
};

enum ge2e_variant { GE2E_SOFTMAX = 0, GE2E_CONTRAST = 1 }; /* paper eq. (6) / eq. (7) */

/* GE2E_FP32: SIMT fp32 FMA everywhere (matches the reference to ~1e-6).
 * GE2E_TF32: similarity and gradient contractions on tcgen05 tensor cores with TF32
 *            operands / fp32 TMEM accumulators (stated tolerance 2e-3).  The softmax row sums are
 *            taken against the fixed shift |w| + b (|cos| <= 1 bounds every logit): exact for
 *            |w| <= 43; beyond that the smallest terms flush to zero (the reference's own
 *            un-stabilised exp(S), s3:120, overflows beyond w + b = 88). */
/* GE2E_FP32_SPLIT: fp32-class accuracy on the tensor cores (reference arithmetic is fp32, s3:57,70).  Every
 *            operand travels as two fp16 planes hi = fp16(x), lo = fp16(x - hi) -- e_hat / c_hat then hold
 *            [rows][2][D] halves in the same bytes as [rows][D] floats (a row's hi plane, then its lo plane: whatever
 *            moves rows -- the all-gather of c_hat, a peer publish -- moves both) -- and every product is the three
 *            kind::f16 MMAs hi.hi + hi.lo + lo.hi with fp32 accumulation (error ~2^-22 per term).  The
 *            softmax probabilities are normalised by a forward launch before the step kernel cuts them into
 *            planes.  Softmax variant, D = 128 or 256, shapes of the tensor-core path only; unlike GE2E_TF32
 *            this is a demand: an uncovered (shape, variant) returns GE2E_ERR_UNSUPPORTED -- ask
 *            ge2e_b200_path() first and fall back to GE2E_FP32.  The planes are written by kernels that read E
 *            16 bytes at a time: E (and dE) must be 16-byte aligned (8 bytes for bf16 / fp16), else GE2E_ERR_UNSUPPORTED (copy an E that
 *            sits at an odd offset of its allocation into fresh storage first). */
/* GE2E_F16:  the hi plane of GE2E_FP32_SPLIT alone: fp16 operands carry the same 11-bit mantissa as TF32 (the
 *            stated tolerance stays 2e-3) at twice its MMA rate, one MMA per product; same kernels, same
 *            row-closing order and the same shape rules as GE2E_FP32_SPLIT (a demand, too).  It pays where the MMAs
 *            dominate (config 4 and its shards); at config 3 the extra forward launch costs more than it saves. */
enum ge2e_precision { GE2E_FP32 = 0, GE2E_TF32 = 1, GE2E_FP32_SPLIT = 2, GE2E_F16 = 3 };

/* Element type of the embeddings E and of their gradient dE (the e_dtype / de_dtype arguments of the _typed entry
 * points; every other buffer of this ABI is fp32 or int32 whatever E is).
 *   E    fp32, bf16 or fp16.  Each element is widened to fp32 exactly when it is loaded; every number after that
 *        load (e_hat, c_hat, cos_diag, the row statistics, loss, dw, db, and dE before its final rounding) is the
 *        one the fp32 call computes for E converted to fp32.  Which kernels run (ge2e_b200_path, the single-kernel
 *        rule, the precisions) depends on the shape only, as for fp32.
 *   dE   fp32 or E's own type (anything else: GE2E_ERR_ARGUMENT).  It is computed in fp32, multiplied by the upstream
 *        gradient grad_out in fp32 and then rounded to its type exactly once (round to nearest even; an fp16 result
 *        beyond its range becomes +-inf, which is what a dynamic loss scaler looks for).  Rounding before the
 *        scaling would flush small fp16 gradients to zero before a loss scale could save them: a caller that runs
 *        the step with grad_out = 1 and applies the real upstream gradient later (ge2e_b200_scale_grads_typed)
 *        keeps dE in fp32 until then.
 * Unknown codes return GE2E_ERR_ARGUMENT before anything is launched.  Alignment: rows of E / dE are read and
 * written four elements at a time where they start at a multiple of four elements (16 bytes for fp32, 8 for the
 * half types); other inputs take the scalar kernels, except under the plane precisions (GE2E_FP32_SPLIT,
 * GE2E_F16), which need that alignment (GE2E_ERR_UNSUPPORTED otherwise). */
enum ge2e_dtype { GE2E_DT_F32 = 0, GE2E_DT_BF16 = 1, GE2E_DT_F16 = 2 };

int ge2e_b200_version(void);
const char* ge2e_b200_strerror(int status);
/* cudaError_t of the last failing CUDA call made by this library on this thread (0 = none). */
int ge2e_b200_last_cuda_error(void);
/* Number of kernels this library has launched (host-side count, all threads). */
unsigned long long ge2e_b200_launch_count(void);
/* Which kernels a (shape, variant, precision) uses: 0 = SIMT fp32 FMA, 1 = tcgen05 TF32, 2 = tcgen05 split
 * fp16 planes (GE2E_FP32_SPLIT), 3 = tcgen05 one fp16 plane (GE2E_F16); the last two answer
 * GE2E_ERR_UNSUPPORTED when the shape / variant is not covered.
 * GE2E_TF32 is a permission, not a demand: shapes the tensor-core path does not cover run on
 * the (more accurate) SIMT kernels.  Negative = bad variant / precision.  The answer depends on the shape
 * only: the plane precisions (2, 3) also need a 16-byte-aligned E (see GE2E_FP32_SPLIT). */
int ge2e_b200_path(int n_local, int n_total, int M, int D, int variant, int precision);
/* Largest M (utterances per speaker) whose backward runs at embedding width D, on every path and alignment;
 * 0 for an unsupported D.  The backward's last stage keeps a speaker's 2 M + 2 rows in 200 KB of shared memory:
 * 199 at D = 128, 99 at D = 256, 49 at D = 512, 24 at D = 1024.  ge2e_b200_forward_backward and
 * ge2e_b200_backward refuse a larger M with GE2E_ERR_UNSUPPORTED before launching anything; a forward alone
 * may still run such a shape.  Host only, no GPU needed. */
int ge2e_b200_max_utterances(int D);
/* Debug: while device_buf is non-NULL the tensor-core kernels run an instrumented instantiation that
 * stamps %globaltimer at its pipeline events into device_buf[grid][3 roles (TMA, MMA, epilogue)][64];
 * NULL switches it off.  kernel: -1 = all, 0 = forward-rows kernel, 1 = step kernel; | 0x100 = also one
 * mark per ring stage in the MMA warp.  Results are unaffected. */
void ge2e_b200_debug_trace(unsigned long long* device_buf, int kernel);
/* Tests / A-B timing: the GE2E_TF32 softmax step runs its first product (S = E_hat C_hat^T) on fp16 copies of the
 * operands -- same 11-bit mantissa, half the shared-memory-bound MMA instructions; the copies are made by one
 * conversion launch in front of the step kernel and live in the workspace -- for shapes of at least 2^26 (local
 * utterance, speaker) pairs (config 4 and its shards; D % 64 == 0).  mode 0 = that rule (initial value), 1 = every
 * supported shape, -1 = never.  Query ge2e_b200_workspace_bytes() AFTER setting it. */
void ge2e_b200_debug_hybrid(int mode);
/* Measurement: while device_buf is non-NULL every CTA of the tensor-core step kernel writes %globaltimer
 * at its start and at its end into device_buf[CTA]{start, end} (two stores per CTA; the production
 * kernel, results unaffected).  max(end) - min(start) is the kernel's duration inside a running step,
 * which CUDA events cannot bracket inside a captured graph. */
void ge2e_b200_debug_stamps(unsigned long long* device_buf);
/* Debug, host only (no GPU needed): the work schedule of the tensor-core step kernel for u_local
 * utterance rows against n_total centroids on max_clusters co-resident clusters of cta_group CTAs.
 * Cluster c works on the pairs [de_begin[c], de_begin[c+1]) of the dE_hat list (pass 1) and [dc_begin[c],
 * dc_begin[c+1]) of the dC_hat list (pass 2) (pair = owner group * units_per_group + stream unit).
 * Arrays need max_clusters + 1 entries.  units = {dE groups, units per dE group, dC groups, units per dC
 * group}; partial = {dE_hat groups are cut between clusters, dC_hat groups are cut}.  Returns the
 * cluster count. */
int ge2e_b200_debug_step_schedule(int u_local, int n_total, int cta_group, int max_clusters,
                                  int* de_begin_host, int* dc_begin_host, int* partial_host,
                                  int* units_host);
/* Debug, host only: the model behind the pass-2 ranges of ge2e_b200_debug_step_schedule (same arguments).
 * Pass 2 of a cluster waits per utterance tile for that tile's row sums, not for the whole grid.  dc_rot_host[c]:
 * cluster c walks its pass-2 range starting that many units in, wrapping around (0 = in order).  finish_host[c]:
 * the model's predicted finish of cluster c, in stream units of work.  model_host = {pass-1 -> pass-2 transition
 * in units, predicted makespan of the same pass-1 cut with a grid barrier between the passes}.  Arrays need
 * max_clusters entries (model_host 2).  Returns the cluster count. */
int ge2e_b200_debug_step_model(int u_local, int n_total, int cta_group, int max_clusters, int* dc_rot_host,
                               double* finish_host, double* model_host);
/* GE2E_OK if the current CUDA device can run this library (sm_100), else GE2E_ERR_DEVICE. */
int ge2e_b200_check_device(void);

/* Scratch needed by ge2e_b200_fwd_rows / ge2e_b200_bwd_rows / ge2e_b200_step_rows for this shape (may
 * be 0; 16-byte aligned).  The workspace must be ZERO-FILLED by the caller before its first use; every
 * call leaves its bookkeeping zero-filled again (stream-K state and grid counters are reset by the last
 * CTA that touches them; the rest is scratch), so a buffer that is kept across calls is zeroed once.
 * One workspace serves one stream.  After a call that FAILED on the device (trap, launch error) zero it
 * again before reuse. */
size_t ge2e_b200_workspace_bytes(int n_local, int n_total, int M, int D, int variant,
                                 int precision);

/* ---- staged entry points (what the sharded autograd function calls) ------------------- */

/* Stage 1 (per rank, local speakers only).
 * Replaces get_centroids (s3:33-38), get_utterance_centroids (s3:95-112) and the
 * leave-one-out cosine cos_same (s3:57).
 *   e_hat[U_local, D]      e / max(|e|, 1e-8)         (TF32: rounded to nearest tf32)
 *   c_hat_local[n_local,D] c_j / max(|c_j|, 1e-8), c_j = mean_i e_ji  (write it straight
 *                          into the rank's slice of the all-gather buffer)
 *   cos_diag[U_local]      cos(e_ji, u_ji), u_ji = (sum_i' e_ji' - e_ji) / (M - 1)
 *   accum[4]               zeroed here: {loss, dw, db, reserved} accumulators            */
int ge2e_b200_prep(const float* E, int n_local, int M, int D, int precision, float* e_hat,
                   float* c_hat_local, float* cos_diag, float* accum, ge2e_stream_t stream);

/* Stage 2: rows of the similarity matrix for the local utterances against ALL centroids,
 * fused with the row loss; S is never written unless sim_out is given.
 * Replaces the expanded cosine + diagonal overwrite + eps (s3:64-79), S = w*cos + b (s3:27)
 * and calc_loss (s3:114-127).
 *   row_stat[U_local]  softmax : log(sum_k exp S_rk + eps)
 *                      contrast: max_{k != j} S_rk
 *   row_kstar[U_local] contrast: argmax (lowest k on ties, -1 if n_total == 1); may be NULL
 *                      for softmax
 *   row_aux[U_local]   softmax : q_r = 1 - p_rj = (sum_{k != j} exp S_rk + eps) / (sum_k exp S_rk
 *                      + eps), accumulated without the diagonal so that the own-speaker
 *                      gradient G_rj = -g q_r does not cancel (the reference's exp(S - lse) - 1
 *                      loses all digits on well-separated speakers); may be NULL for contrast
 *   loss_accum         += sum of the local rows' losses (zeroed by ge2e_b200_prep)
 *   per_row_out        optional [U_local] per-embedding loss (s3:121)
 *   sim_out            optional [U_local, n_total] cos + eps (what get_cos_sim returns)
 *   dE_hat, row_scale  optional, both or neither: "a backward will follow".  Where the softmax loss
 *                      runs on tensor cores (ge2e_b200_path() == 1) the forward is then the rows pass
 *                      of the step kernel: S is computed once, P = exp(S - (|w| + b)) feeds the row
 *                      sums AND, from tensor memory, the contraction P . C_hat, so the forward leaves
 *                        dE_hat[U_local, D]  UN-NORMALISED off-diagonal gradient rows
 *                        row_scale[U_local]  w exp(|w| + b - lse_r): the true row is
 *                                            g * row_scale[r] * dE_hat[r]   (applied by bwd_finalize)
 *                      and ge2e_b200_bwd_rows has only the centroid pass left.  On every other path the
 *                      two pointers are ignored (nothing is written).                                 */
int ge2e_b200_fwd_rows(const float* e_hat, const float* c_hat_all, const float* cos_diag,
                       int n_local, int n_total, int spk_offset, int M, int D,
                       const float* w, const float* b, float eps, int variant, int precision,
                       float* row_stat, int32_t* row_kstar, float* row_aux, float* loss_accum,
                       float* per_row_out, float* sim_out, float* dE_hat, float* row_scale,
                       void* workspace, size_t workspace_bytes, ge2e_stream_t stream);

/* Stage 3: gradient wrt the normalised operands, S recomputed on the fly (never stored).
 * Replaces the autograd graph of s3:57-79 / s3:114-127 (SURVEY 8(a-bis) items 7-9).
 *   dE_hat[U_local, D]         sum_{k != j} w G_rk c_hat_k          (off-diagonal part)
 *   dC_hat_partial[n_total, D] sum_{local r, k != j(r)} w G_rk e_hat_r  (zeroed inside;
 *                              reduce-scatter it across ranks when sharded)
 *   dwdb_accum[2]              = {dw, db} of the local rows (zeroed inside, then accumulated)
 *   row_scale                  the forward's row_scale when ge2e_b200_fwd_rows was given dE_hat /
 *                              row_scale on the tensor-core softmax path: dE_hat is then left as the
 *                              forward wrote it and only dC_hat_partial, dw, db are produced.  NULL:
 *                              dE_hat is computed here (on the SIMT kernels where the tensor-core
 *                              forward did not prepare it).                                        */
int ge2e_b200_bwd_rows(const float* e_hat, const float* c_hat_all, const float* cos_diag,
                       const float* row_stat, const int32_t* row_kstar, const float* row_aux,
                       const float* row_scale,
                       int n_local, int n_total, int spk_offset, int M, int D, const float* w,
                       const float* b, float eps, int variant, int precision,
                       const float* grad_out, float* dE_hat, float* dC_hat_partial,
                       float* dwdb_accum, void* workspace, size_t workspace_bytes,
                       ge2e_stream_t stream);

/* Stage 4 (per rank, local speakers): diagonal (leave-one-out) term, the three
 * normalisation Jacobians and the centroid fan-out (SURVEY 8(a-bis) items 9-11).
 *   dC_hat_local[n_local, D]  this rank's rows of the (reduced) dC_hat
 *   row_scale                 NULL, or the forward's row_scale (dE_hat rows are un-normalised, see
 *                             ge2e_b200_fwd_rows): row r of dE_hat counts g * row_scale[r] times
 *   dE[U_local, D]            gradient wrt the raw embeddings                            */
int ge2e_b200_bwd_finalize(const float* E, const float* dE_hat, const float* dC_hat_local,
                           const float* cos_diag, const float* row_stat, const float* row_aux,
                           const float* row_scale, int n_local, int M, int D, const float* w,
                           const float* b, float eps, int variant, const float* grad_out, float* dE,
                           ge2e_stream_t stream);

/* Stages 2 + 3 in one call, for a step whose forward and backward are issued together (a captured
 * training step; the sharded step between its all-gather and its reduce-scatter):
 * ge2e_b200_fwd_rows followed by ge2e_b200_bwd_rows with the same buffers.  Where the softmax loss runs
 * on tensor cores this is ONE persistent kernel: rows pass (loss, row statistics, un-normalised dE_hat),
 * a grid-wide barrier, centroid pass (dC_hat_partial, dw, db): 8 U N D issued flops for 6 U N D
 * algorithmic, S never stored.
 *   accum[4]   {loss, dw, db, -}: += (zeroed by ge2e_b200_prep, which must precede this call)
 *   row_scale  [U_local] out: pass it to ge2e_b200_bwd_finalize when ge2e_b200_path() == 1 and the
 *              variant is softmax, NULL otherwise                                              */
int ge2e_b200_step_rows(const float* e_hat, const float* c_hat_all, const float* cos_diag, int n_local,
                        int n_total, int spk_offset, int M, int D, const float* w, const float* b,
                        float eps, int variant, int precision, const float* grad_out, float* row_stat,
                        int32_t* row_kstar, float* row_aux, float* row_scale, float* accum,
                        float* dE_hat, float* dC_hat_partial, void* workspace, size_t workspace_bytes,
                        ge2e_stream_t stream);

/* ---- speaker-sharded step over PEER MEMORY (one NVLink / NVSwitch domain, <= 8 ranks) ----------
 * The two exchange steps of the sharded loss (SURVEY 8(e)) without collective kernels: the ranks map each
 * other's buffers (CUDA peer access / symmetric memory; the Python layer uses
 * torch.distributed._symmetric_memory) and the kernels store / add across NVLink themselves.
 *   all-gather of c_hat      ge2e_b200_peer_publish: src[n_floats] -- this rank's slice of c_hat, the rows prep
 *                            just wrote into its own c_hat_all -- is stored to dst_host[0 .. n_dst) (a HOST
 *                            array of device pointers: the same slice of every PEER's c_hat_all), or, with
 *                            multicast != 0 and n_dst == 1, to ONE multicast address of the NVSwitch domain
 *                            (multimem.st: one store leaves the GPU, the switch replicates it to every rank);
 *                            zero[zero_floats] (nullable: this rank's dC_local) is cleared.  The same call
 *                            publishes a rank's {loss, dw, db} partials into the peers' scalar tables;
 *   -- cross-rank barrier (caller: e.g. the symmetric-memory handle's barrier) --
 *   reduce-scatter of dC_hat ge2e_b200_step_rows_peers: ge2e_b200_step_rows whose centroid pass reduce-adds
 *                            every accumulator tile straight into the OWNER rank's rows (TMA
 *                            cp.reduce.async.bulk into peer memory: the fp32 add happens at the owner's L2)
 *                            -- dC_owner_host[r] = rank r's dC_local[n_total / n_ranks, D], a HOST array of
 *                            n_ranks device pointers, this rank's own included -- instead of into a
 *                            full-height partial that a reduce-scatter sums afterwards;
 *   -- cross-rank barrier --, then ge2e_b200_bwd_finalize on dC_local as usual.
 * Tensor-core softmax shapes with (n_total / n_ranks) % 128 == 0 only (GE2E_ERR_UNSUPPORTED otherwise: use
 * ge2e_b200_step_rows + a reduce-scatter).  The {loss, dw, db} partials of accum[] are exchanged by the
 * caller (ShardedGE2EPlan publishes them into a [ranks, 4] table in front of the second barrier).
 * The contrast loss takes ge2e_b200_fwd_rows, then ge2e_b200_contrast_bwd_rows_peers (below, with the per-utterance
 * entry points) in place of ge2e_b200_step_rows_peers. */
int ge2e_b200_peer_publish(const float* src, float* const* dst_host, int n_dst, int multicast,
                           long long n_floats, float* zero, long long zero_floats, ge2e_stream_t stream);
int ge2e_b200_step_rows_peers(const float* e_hat, const float* c_hat_all, const float* cos_diag, int n_local,
                              int n_total, int spk_offset, int M, int D, const float* w, const float* b,
                              float eps, int variant, int precision, const float* grad_out, float* row_stat,
                              int32_t* row_kstar, float* row_aux, float* row_scale, float* accum,
                              float* dE_hat, float* const* dC_owner_host, int n_ranks, void* workspace,
                              size_t workspace_bytes, ge2e_stream_t stream);

/* The trainer's post-loss tail for the two loss parameters, on the device (SURVEY 8(f) row 1;
 * replaces `torch.nn.utils.clip_grad_norm_(self.ge2e_loss.parameters(), 1.0)` and the loss
 * parameter group's share of `self.optimizer.step()` (plain SGD), s4_train_embed_model.py:202-203,
 * :35-42).  clip_grad_norm_ semantics: total = sqrt(dw^2 + db^2); coef = min(1, max_norm /
 * (total + 1e-6)); dw, db are scaled by coef IN PLACE (as the reference leaves them), then
 * w -= lr * dw, b -= lr * db.  total_norm (nullable, device) receives the unclipped norm, the value
 * clip_grad_norm_ returns.  All pointers are device pointers to single floats.  Enqueue it after the
 * backward on the same stream; one one-thread kernel, launched under the previous kernel's tail. */
int ge2e_b200_scale_bias_sgd(float* w, float* b, float* dw, float* db, float max_norm, float lr,
                             float* total_norm, ge2e_stream_t stream);

/* The whole step of the trainer in one call (s4_train_embed_model.py:196 + :200: `loss =
 * self.ge2e_loss(embeddings); loss.backward()`): ge2e_b200_prep_indexed, ge2e_b200_step_rows and
 * ge2e_b200_bwd_finalize_indexed with the same buffers (row_index nullable; accum[0] = loss,
 * accum[1] = dw, accum[2] = db; grad_out = device scalar, the upstream gradient).
 * Batches of the reference's own size -- N <= 128 speakers, M <= 16, D <= 256, i.e. its training
 * (64 x 10) and test (4 x 8) shapes, where five dependent launches are mostly latency -- run as ONE
 * kernel (the kernel itself supports N <= 128, see ge2e_b200_debug_small_step):
 * one CTA per speaker, every stage separated by grid-wide barriers (all CTAs are co-resident; up to 8 speakers
 * the grid is one thread-block cluster), centroid gradients added at the L2 (one bulk reduce-add per CTA; rows
 * that are not whole 16-byte multiples go through the workspace in a fixed order instead).  Those shapes
 * need ge2e_b200_step_workspace_bytes() bytes of workspace (>= ge2e_b200_workspace_bytes()); only its
 * first 256 bytes have to be zero on entry and are zero again on exit, the rest is scratch.
 * ge2e_b200_step_launches() = 1 when the single-kernel path is taken for the shape, else 0. */
size_t ge2e_b200_step_workspace_bytes(int N, int M, int D, int variant, int precision);
/* Debug / tests: which shapes take the single-kernel step.  0 = none, 1 = those where it was measured
 * faster than the pipeline (all of them since round 2: N <= 128; default), 2 = every shape the kernel supports (N <= 128, M <= 16, D <= 256).
 * Initial value 1.  Query sizes / launches AFTER setting it. */
void ge2e_b200_debug_small_step(int mode);
int ge2e_b200_step_launches(int N, int M, int D, int variant, int precision);
/* The step's gradients for another upstream gradient: the loss is linear in it, so a step that ran with
 * grad_out = 1 (what an eager `loss = crit(E)` does when it computes the whole step in its forward) is finished by
 * dE_out[n] = g * dE_in[n], dwdb_out[2] = g * dwdb_in[2] -- one launch (`loss.backward()`, s4:200). */
int ge2e_b200_scale_grads(const float* dE_in, float* dE_out, long long n, const float* dwdb_in, float* dwdb_out,
                          const float* grad_out, ge2e_stream_t stream);
/* The same with dE_out of type de_dtype (ge2e_dtype): dE_in stays fp32, each g * dE_in[n] is rounded once. */
int ge2e_b200_scale_grads_typed(const float* dE_in, void* dE_out, int de_dtype, long long n, const float* dwdb_in,
                                float* dwdb_out, const float* grad_out, ge2e_stream_t stream);
int ge2e_b200_forward_backward(const float* E, const int32_t* row_index, int N, int M, int D, const float* w,
                               const float* b, float eps, int variant, int precision, const float* grad_out,
                               float* e_hat, float* c_hat, float* cos_diag, float* row_stat, int32_t* row_kstar,
                               float* row_aux, float* row_scale, float* accum, float* dE_hat, float* dC_hat,
                               float* dE, void* workspace, size_t workspace_bytes, ge2e_stream_t stream);

/* Batch assembly from a device-resident spectrogram bank (SURVEY 8(f) row 4;
 * s1_dataset_loader.py:59-77 `spr_utters[utter_idx][:, clip:clip + L, :]`, the DataLoader's collate,
 * and s4_train_embed_model.py:176-186 reshape + `mel_db_batch[perm]`): a cropped utterance is one
 * contiguous span of its speaker's [utts, frames, mels] array, so the model's input batch is
 *   out[r, 0:span] = bank[src_off[r] : src_off[r] + span],  r = 0 .. rows-1   (span = L * mels)
 * with src_off[rows] (device, int64, element offsets) computed by the host from the drawn utterance
 * indices, crop start and row permutation.  offsets_aligned != 0 promises that every offset is a
 * multiple of 4 floats (16-byte vector path when span % 4 == 0 as well); 0 selects the scalar kernel.
 * fp32 in, fp32 out, bit-exact copy. */
int ge2e_b200_gather_spans(const float* bank, const long long* src_off, int rows, long long span, int offsets_aligned,
                           float* out, ge2e_stream_t stream);

/* Model tail feeding the loss (SURVEY 8(f) row 2; s2_model_GE2E_loss_speach_embed.py:28-34:
 * `x = x[:, x.size(1) - 1]; x = self.projection(x); x = x / torch.norm(x, dim=1).unsqueeze(1)`).
 * One tcgen05 (TF32, fp32 accumulate) kernel: E = normalise_rows(X W^T + bias).
 *   X[U, H]      device fp32, row r at X + r * x_row_stride floats (the last-frame select of the
 *                LSTM output [U, frames, H] is x_row_stride = frames * H with X pointing at the last
 *                frame of row 0); H % 4 == 0, x_row_stride % 4 == 0, 16-byte aligned
 *   W[D, H]      nn.Linear weight (row-major, contiguous), D in {64, 128, 256}
 *   bias[D]      nullable
 *   E[U, D]      unit rows (no epsilon, as the reference: a zero row gives NaN)
 *   inv_norm[U]  1 / ||X W^T + bias|| per row, kept for the backward (nullable)
 * GE2E_ERR_UNSUPPORTED for other shapes / alignments. */
int ge2e_b200_embed_tail_fwd(const float* X, long long x_row_stride, const float* W, const float* bias, int U,
                             int H, int D, float* E, float* inv_norm, ge2e_stream_t stream);
/* Backward of the normalisation and the bias: dY = (dE - E (E . dE)) * inv_norm (row-wise),
 * dbias[D] = column sums of dY (nullable; zeroed by the call). */
int ge2e_b200_embed_tail_bwd_rows(const float* dE, const float* E, const float* inv_norm, int U, int D, float* dY,
                                  float* dbias, ge2e_stream_t stream);
/* The two gradient GEMMs of the Linear layer (what autograd runs under s2_model_GE2E_loss_speach_embed.py:31),
 * on tcgen05 with TF32 operands / fp32 accumulation like the forward:
 *   dX[U, H] = dY[U, D] W[D, H]       rows dx_row_stride floats apart: the gradient of the last-frame select is
 *                                     written straight into the last frame of a zeroed [U, frames, H] tensor
 *   dW[D, H] = dY^T X[U, H]           X rows x_row_stride apart (as in the forward); the sum over U is split over
 *                                     CTAs and added at the L2 (dW is zeroed by the call)
 * dX or dW may be NULL (that product is skipped).  Needs H % 32 == 0, D in {64, 128, 256}, strides % 4 == 0,
 * 16-byte aligned pointers: ..._supported() returns 1 where this holds, GE2E_ERR_UNSUPPORTED otherwise (the host
 * layer then issues plain library GEMMs). */
int ge2e_b200_embed_tail_bwd_gemms_supported(int U, int H, int D, long long x_row_stride, long long dx_row_stride);
int ge2e_b200_embed_tail_bwd_gemms(const float* dY, const float* W, const float* X, long long x_row_stride, int U,
                                   int H, int D, float* dX, long long dx_row_stride, float* dW, ge2e_stream_t stream);

/* EER sweep counts (SURVEY 8(f) row 3; s5_eval_model.py:57-89: `S_thres = S > thres`,
 * `np.sum(S_thres[i])`, `np.sum(S_thres[i, :, i])` for 50 thresholds).  One pass over the float32
 * similarity matrix sim[N, M, N] (device) for all T thresholds at once:
 *   thresholds[T]  device, float32, ASCENDING (duplicates allowed), 1 <= T <= 1024
 *   accept_all[T]  device int64: entries of sim greater than thresholds[t]
 *   accept_own[T]  device int64: the same over the own-speaker entries sim[j, :, j]
 *   scratch        device, ge2e_b200_threshold_counts_scratch_bytes(T) bytes (zeroed by the call)
 * FAR / FRR / EER (s5:80-97) are a few scalar operations on these counts and stay on the host
 * (speaker_embedding_ge2e_loss_b200/evaluation.py).  Comparisons are float32 `>` as in numpy; a NaN
 * entry exceeds no threshold.  Integer results, bit-exact. */
size_t ge2e_b200_threshold_counts_scratch_bytes(int T);
int ge2e_b200_threshold_counts(const float* sim, int N, int M, const float* thresholds, int T,
                               long long* accept_all, long long* accept_own, void* scratch,
                               size_t scratch_bytes, ge2e_stream_t stream);

/* ---- single-device conveniences (n_local == n_total) ---------------------------------- */

/* GE2ELoss.forward (s3:19-30): prep + fwd_rows.  loss = accum[0].  dE_hat / row_scale: NULL for a
 * forward that no backward follows, else buffers [N*M, D] / [N*M] to hand to ge2e_b200_backward (see
 * ge2e_b200_fwd_rows). */
int ge2e_b200_forward(const float* E, int N, int M, int D, const float* w, const float* b,
                      float eps, int variant, int precision, float* e_hat, float* c_hat,
                      float* cos_diag, float* row_stat, int32_t* row_kstar, float* row_aux,
                      float* accum, float* dE_hat, float* row_scale, void* workspace,
                      size_t workspace_bytes, ge2e_stream_t stream);

/* loss.backward() (s4:200): bwd_rows + bwd_finalize.  dw = accum[1], db = accum[2].  dE_hat /
 * row_scale: the buffers the forward was given (row_scale NULL if it was given none). */
int ge2e_b200_backward(const float* E, const float* e_hat, const float* c_hat,
                       const float* cos_diag, const float* row_stat, const int32_t* row_kstar,
                       const float* row_aux, const float* row_scale, int N, int M, int D, const float* w,
                       const float* b, float eps, int variant, int precision, const float* grad_out,
                       float* dE_hat, float* dC_hat, float* accum, float* dE, void* workspace,
                       size_t workspace_bytes, ge2e_stream_t stream);

/* ---- row-indexed variants (SURVEY 8(f) row 1: the trainer's unperm gather) ------------- */

/* The trainer shuffles the utterances before the embedder and undoes the shuffle right before the
 * loss: `embeddings = embeddings[unperm]; embeddings.reshape(N, M, D)` (s4_train_embed_model.py:
 * 177-192), a row gather whose autograd backward is a row scatter.  The _indexed entry points fold
 * both into the loss: E (and dE) stay in the embedder's row order, logical row r = [speaker][utterance]
 * lives at physical row row_index[r] (int32, device, a permutation of [0, n_local * M)).  Prep reads
 * through the index, finalize writes dE through it; everything in between is unchanged.
 * row_index == NULL is the plain call.                                                     */
int ge2e_b200_prep_indexed(const float* E, const int32_t* row_index, int n_local, int M, int D,
                           int precision, float* e_hat, float* c_hat_local, float* cos_diag,
                           float* accum, ge2e_stream_t stream);
int ge2e_b200_bwd_finalize_indexed(const float* E, const int32_t* row_index, const float* dE_hat,
                                   const float* dC_hat_local, const float* cos_diag,
                                   const float* row_stat, const float* row_aux, const float* row_scale,
                                   int n_local, int M, int D, const float* w, const float* b, float eps,
                                   int variant, const float* grad_out, float* dE, ge2e_stream_t stream);
int ge2e_b200_forward_indexed(const float* E, const int32_t* row_index, int N, int M, int D,
                              const float* w, const float* b, float eps, int variant, int precision,
                              float* e_hat, float* c_hat, float* cos_diag, float* row_stat,
                              int32_t* row_kstar, float* row_aux, float* accum, float* dE_hat,
                              float* row_scale, void* workspace, size_t workspace_bytes,
                              ge2e_stream_t stream);
int ge2e_b200_backward_indexed(const float* E, const int32_t* row_index, const float* e_hat,
                               const float* c_hat, const float* cos_diag, const float* row_stat,
                               const int32_t* row_kstar, const float* row_aux, const float* row_scale,
                               int N, int M, int D,
                               const float* w, const float* b, float eps, int variant, int precision,
                               const float* grad_out, float* dE_hat, float* dC_hat, float* accum,
                               float* dE, void* workspace, size_t workspace_bytes,
                               ge2e_stream_t stream);

/* ---- embeddings of another element type (ge2e_dtype) ------------------------------------
 * The _indexed entry points (row_index nullable) with E of type e_dtype and dE of type de_dtype.  The plain and
 * _indexed entry points are these with GE2E_DT_F32 for both.  All other buffers are fp32 / int32 as above. */
int ge2e_b200_prep_typed(const void* E, int e_dtype, const int32_t* row_index, int n_local, int M, int D,
                         int precision, float* e_hat, float* c_hat_local, float* cos_diag, float* accum,
                         ge2e_stream_t stream);
int ge2e_b200_bwd_finalize_typed(const void* E, int e_dtype, const int32_t* row_index, const float* dE_hat,
                                 const float* dC_hat_local, const float* cos_diag, const float* row_stat,
                                 const float* row_aux, const float* row_scale, int n_local, int M, int D,
                                 const float* w, const float* b, float eps, int variant, const float* grad_out,
                                 void* dE, int de_dtype, ge2e_stream_t stream);
int ge2e_b200_forward_typed(const void* E, int e_dtype, const int32_t* row_index, int N, int M, int D,
                            const float* w, const float* b, float eps, int variant, int precision, float* e_hat,
                            float* c_hat, float* cos_diag, float* row_stat, int32_t* row_kstar, float* row_aux,
                            float* accum, float* dE_hat, float* row_scale, void* workspace, size_t workspace_bytes,
                            ge2e_stream_t stream);
int ge2e_b200_backward_typed(const void* E, int e_dtype, const int32_t* row_index, const float* e_hat,
                             const float* c_hat, const float* cos_diag, const float* row_stat,
                             const int32_t* row_kstar, const float* row_aux, const float* row_scale, int N, int M,
                             int D, const float* w, const float* b, float eps, int variant, int precision,
                             const float* grad_out, float* dE_hat, float* dC_hat, float* accum, void* dE,
                             int de_dtype, void* workspace, size_t workspace_bytes, ge2e_stream_t stream);
int ge2e_b200_forward_backward_typed(const void* E, int e_dtype, const int32_t* row_index, int N, int M, int D,
                                     const float* w, const float* b, float eps, int variant, int precision,
                                     const float* grad_out, float* e_hat, float* c_hat, float* cos_diag,
                                     float* row_stat, int32_t* row_kstar, float* row_aux, float* row_scale,
                                     float* accum, float* dE_hat, float* dC_hat, void* dE, int de_dtype,
                                     void* workspace, size_t workspace_bytes, ge2e_stream_t stream);

/* ---- per-utterance losses (reduction "none") ---------------------------------------------
 * L_r, the loss of utterance row r in logical [speaker][utterance] order (calc_loss's per_embedding_loss, s3:121):
 *   softmax  log(sum_k exp S_rk + eps) - S_rj        contrast  1 - sigmoid(S_rj) + max_{k != j} sigmoid(S_rk)
 * ge2e_b200_forward_per_row_typed: ge2e_b200_forward_typed that also writes per_row[N*M] (device, required);
 *   accum[0] is still the sum.
 * ge2e_b200_backward_per_row_typed: ge2e_b200_backward_typed for the upstream gradient grad_rows[N*M] (device, logical
 *   order, required; any values, negative and zero included) in place of the scalar grad_out:
 *   dE = sum_r grad_rows[r] dL_r / dE, accum[1] = dw, accum[2] = db likewise; dE is rounded to de_dtype once.
 * A NULL per_row / grad_rows returns GE2E_ERR_ARGUMENT before anything is launched.  The upstream gradient is known
 * only after the forward, so the forward and the backward are separate launches.  On the shapes where
 * ge2e_b200_forward_backward runs the single-kernel step (ge2e_b200_step_launches() == 1, same
 * ge2e_b200_debug_small_step rule) and the workspace has at least ge2e_b200_step_workspace_bytes() bytes, each is
 * ONE kernel -- that step cut after the row losses: the forward runs prep and the losses; the backward re-reads E,
 * recomputes the cosines from e_hat / c_hat, forms w G from grad_rows and the row statistics and runs the rest of
 * the step.  Otherwise (a workspace of ge2e_b200_workspace_bytes(), every other shape) they run the staged kernels.
 * Both forms leave and read the same forward outputs, so either forward pairs with either backward.  The
 * whole-step-in-forward scheme (ge2e_b200_forward_backward with grad_out = 1, then ge2e_b200_scale_grads) has no
 * per-row form.  The speaker-sharded forward writes per_row through ge2e_b200_fwd_rows; its backward stages follow. */
int ge2e_b200_forward_per_row_typed(const void* E, int e_dtype, const int32_t* row_index, int N, int M, int D,
                                    const float* w, const float* b, float eps, int variant, int precision, float* e_hat,
                                    float* c_hat, float* cos_diag, float* row_stat, int32_t* row_kstar, float* row_aux,
                                    float* accum, float* dE_hat, float* row_scale, float* per_row, void* workspace,
                                    size_t workspace_bytes, ge2e_stream_t stream);
int ge2e_b200_backward_per_row_typed(const void* E, int e_dtype, const int32_t* row_index, const float* e_hat,
                                     const float* c_hat, const float* cos_diag, const float* row_stat,
                                     const int32_t* row_kstar, const float* row_aux, const float* row_scale, int N,
                                     int M, int D, const float* w, const float* b, float eps, int variant,
                                     int precision, const float* grad_rows, float* dE_hat, float* dC_hat, float* accum,
                                     void* dE, int de_dtype, void* workspace, size_t workspace_bytes,
                                     ge2e_stream_t stream);

/* Per-utterance losses over speaker shards.  Rank q's objective term is sum_r grad_rows_q[r] L_r over its own rows;
 * the sum over ranks is differentiated, so dE_local also carries what the other ranks' rows send through this rank's
 * centroids, and dw / db are global once the ranks' partials are summed.  grad_rows: device, [n_local * M], this
 * rank's rows in logical [speaker][utterance] order, any values.  NULL grad_rows returns GE2E_ERR_ARGUMENT before
 * anything is launched.
 *   ge2e_b200_bwd_rows_per_row             ge2e_b200_bwd_rows with grad_rows in place of grad_out: on the tensor-core
 *                                          softmax path with the forward's row_scale the lone centroid pass (dC_hat
 *                                          partial [n_total, D] and this rank's {dw, db}), else the SIMT kernels.
 *                                          The caller then reduce-scatters dC_hat and all-reduces {dw, db}.
 *   ge2e_b200_bwd_finalize_per_row_typed   ge2e_b200_bwd_finalize_typed with grad_rows: row r of an un-normalised
 *                                          dE_hat counts grad_rows[r] * row_scale[r] times; dE in de_dtype.
 *   ge2e_b200_bwd_rows_peers_per_row       the centroid pass of ge2e_b200_step_rows_peers alone, for grad_rows: every
 *                                          dC_hat accumulator tile is reduce-added into the owner rank's dC_local
 *                                          (dC_owner_host, n_ranks as there; the owners cleared their rows before the
 *                                          cross-rank barrier in front of this call), dwdb_accum[2] receives this
 *                                          rank's {dw, db} (overwritten).  row_scale (required) says that the
 *                                          forward (ge2e_b200_fwd_rows with dE_hat + row_scale) prepared dE_hat.
 *                                          GE2E_ERR_SHAPE for n_ranks outside 2..GE2E_MAX_PEERS or n_local * n_ranks
 *                                          != n_total; GE2E_ERR_UNSUPPORTED where ge2e_b200_step_rows_peers refuses
 *                                          (contrast, GE2E_FP32, owner rows not whole 128-row tiles);
 *                                          GE2E_ERR_ARGUMENT for a NULL or misaligned owner pointer.  Every refusal
 *                                          returns before anything is launched or written. */
int ge2e_b200_bwd_rows_per_row(const float* e_hat, const float* c_hat_all, const float* cos_diag,
                               const float* row_stat, const int32_t* row_kstar, const float* row_aux,
                               const float* row_scale, int n_local, int n_total, int spk_offset, int M, int D,
                               const float* w, const float* b, float eps, int variant, int precision,
                               const float* grad_rows, float* dE_hat, float* dC_hat_partial, float* dwdb_accum,
                               void* workspace, size_t workspace_bytes, ge2e_stream_t stream);
int ge2e_b200_bwd_finalize_per_row_typed(const void* E, int e_dtype, const int32_t* row_index, const float* dE_hat,
                                         const float* dC_hat_local, const float* cos_diag, const float* row_stat,
                                         const float* row_aux, const float* row_scale, int n_local, int M, int D,
                                         const float* w, const float* b, float eps, int variant,
                                         const float* grad_rows, void* dE, int de_dtype, ge2e_stream_t stream);
int ge2e_b200_bwd_rows_peers_per_row(const float* e_hat, const float* c_hat_all, const float* cos_diag,
                                     const float* row_stat, const float* row_aux, const float* row_scale, int n_local,
                                     int n_total, int spk_offset, int M, int D, const float* w, const float* b,
                                     float eps, int variant, int precision, const float* grad_rows, float* dE_hat,
                                     float* dwdb_accum, float* const* dC_owner_host, int n_ranks, void* workspace,
                                     size_t workspace_bytes, ge2e_stream_t stream);

/* The contrast loss over peer memory (ge2e_b200_step_rows_peers keeps refusing it: its backward is no contraction).
 * After ge2e_b200_fwd_rows has written row_stat / row_kstar, the backward rows stage is one gather / scatter kernel:
 * dE_hat row r = w G_n c_hat[k*] (zero where k* < 0), and w G_n e_hat_r is added straight into centroid k*'s row of
 * its owner rank, row k* % (n_total / n_ranks) of dC_owner_host[k* / (n_total / n_ranks)] (a HOST array of n_ranks
 * device pointers, every rank's dC_local, this rank's own included; the owners cleared their rows before the
 * cross-rank barrier in front of this call).  The adds are reductions at the owner's memory: red.global.add.v4.f32
 * where D % 4 == 0, scalar ones otherwise.  dwdb_accum[2] receives this rank's {dw, db} (overwritten); the caller
 * exchanges them (ShardedGE2EPlan: its scalar table).  GE2E_FP32 and GE2E_TF32 run the same kernel (it reads
 * c_hat_all in fp32 either way); n_local need not be a multiple of 128.
 *   ge2e_b200_contrast_bwd_rows_peers          the scalar upstream gradient grad_out (device, one float)
 *   ge2e_b200_contrast_bwd_rows_peers_per_row  grad_rows[n_local * M] in its place (reduction="none")
 * Refusals, every one before anything is launched or written: GE2E_ERR_ARGUMENT for a NULL pointer (grad_rows on the
 * per-row form included) or a NULL owner pointer, or one not 16-byte aligned where D % 4 == 0 (4-byte otherwise);
 * GE2E_ERR_SHAPE for n_ranks outside 2..GE2E_MAX_PEERS or n_local * n_ranks != n_total; GE2E_ERR_UNSUPPORTED for
 * GE2E_FP32_SPLIT / GE2E_F16 (contrast has no fp16-plane path); a bad shape as ge2e_b200_bwd_rows. */
int ge2e_b200_contrast_bwd_rows_peers(const float* e_hat, const float* c_hat_all, const float* cos_diag,
                                      const float* row_stat, const int32_t* row_kstar, int n_local, int n_total,
                                      int spk_offset, int M, int D, const float* w, const float* b, float eps,
                                      int precision, const float* grad_out, float* dE_hat, float* dwdb_accum,
                                      float* const* dC_owner_host, int n_ranks, ge2e_stream_t stream);
int ge2e_b200_contrast_bwd_rows_peers_per_row(const float* e_hat, const float* c_hat_all, const float* cos_diag,
                                              const float* row_stat, const int32_t* row_kstar, int n_local,
                                              int n_total, int spk_offset, int M, int D, const float* w,
                                              const float* b, float eps, int precision, const float* grad_rows,
                                              float* dE_hat, float* dwdb_accum, float* const* dC_owner_host,
                                              int n_ranks, ge2e_stream_t stream);

/* ---- static helpers of the reference class (used by s5_eval_model.py:42-43) ----------- */

/* get_centroids (s3:33-38): C[N, D] = mean over utterances. */
int ge2e_b200_centroids(const float* E, int N, int M, int D, float* C, ge2e_stream_t stream);
/* get_utterance_centroids (s3:95-112): Uc[N, M, D]. */
int ge2e_b200_utterance_centroids(const float* E, int N, int M, int D, float* Uc,
                                  ge2e_stream_t stream);
/* Y[rows, D] = X / max(|X_row|, 1e-8): lets get_cos_sim (s3:41-80) accept caller-supplied
 * centroids the way the reference's static method does (s5_eval_model.py:43). */
int ge2e_b200_normalize_rows(const float* X, int rows, int D, float* Y, ge2e_stream_t stream);
/* calc_loss (s3:114-127) on a caller-supplied similarity matrix S[N, M, N]. */
int ge2e_b200_calc_loss(const float* S, int N, int M, float eps, int variant, float* loss,
                        float* per_row, ge2e_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GE2E_B200_H_ */
