/* cals_b200.h -- C ABI of the B200-native CP-CALS hot path.
 *
 * The reference (HPAC/CP-CALS) has no FFI of its own: its accelerator seam is the C++ API
 *     cals::cp_cals(const Tensor&, KtensorQueue&, CalsParams&)      reference include/cals.h:196
 *     cals::jk_cp_cals(const Tensor&, vector<Ktensor>&, CalsParams&) reference include/cals.h:198
 * with `CalsParams::cuda` (include/cals.h:150) routing the MTTKRP to cuBLAS + one kernel
 * (src/utils/mttkrp.cpp:156-162,233-265,341-420; src/utils/khatri_rao.cu:40).  This header is the thin C layer that
 * the C++ host code of this repository (include/cals.h ... , cp-cals_b200/host/) calls instead; a maintainer of the
 * reference would bind exactly these entry points from src/cals.cpp (see INTEGRATION.md).
 *
 * Conventions: every function returns 0 on success, non-zero on error (message via cals_b200_last_error); no
 * exceptions cross this boundary; all pointers are HOST pointers unless the name ends in _dev; all matrices are
 * FP64 column-major; the tensor is column-major with mode 0 fastest (reference src/tensor.cpp:143-180).  One
 * context per caller thread.  There is no CPU fallback: without a CUDA device every call fails loudly.
 */
#ifndef CALS_B200_H
#define CALS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cals_b200_ctx cals_b200_ctx;

/* flags for cals_b200_configure (CalsParams::force_max_iter / always_evict_first, reference include/cals.h:158-159) */
#define CALS_B200_FORCE_MAX_ITER 1u
#define CALS_B200_ALWAYS_EVICT_FIRST 2u
/* CalsParams::update_method == NNLS (reference include/utils/update.h:8, src/utils/update.cpp:61-176): non-negative
 * factors by a row-wise active-set solve instead of the Cholesky solve */
#define CALS_B200_NNLS 4u

/* MTTKRP kernel variants (test hook / tuning knob; the product default is CALS_B200_MTTKRP_DMMA) */
#define CALS_B200_MTTKRP_DMMA 0  /* TMA + mbarrier pipeline, FP64 tensor-core mma.sync, stream-K partials */
#define CALS_B200_MTTKRP_NAIVE 1 /* one thread per output element; cross-check only */

/* Filled by cals_b200_run: the fields of the reference's CalsReport (include/cals.h:27-63) that the path produces. */
typedef struct cals_b200_report {
  uint64_t iter;             /* CalsReport::iter: global CALS iterations executed */
  uint64_t n_ktensors;       /* CalsReport::n_ktensors */
  uint64_t ktensor_comp_sum; /* CalsReport::ktensor_comp_sum */
  double x_norm;             /* CalsReport::X_norm */
  double total_time;         /* seconds, host wall clock around the device loop (CalsReport::total_time) */
  double device_ms;          /* CUDA-event time of the whole iteration loop */
  double mttkrp_ms;          /* CUDA-event time summed over the MTTKRP kernels (0 unless timing enabled) */
  double update_ms;          /* CUDA-event time summed over the per-model update/fit kernels (idem) */
  uint64_t mttkrp_launches;  /* number of MTTKRP kernel launches */
  uint64_t kernel_launches;  /* all kernels launched by this run */
  double mttkrp_flops;       /* algorithmic flop executed by the MTTKRPs: sum over launches of 2*nX*C */
  double exchange_ms;        /* sliced tensor + timing: CUDA-event time summed over the peer-memory exchange kernels
                                (barrier wait + NVLink pulls); it is part of mttkrp_ms as well */
  /* 3-mode tensors held whole by one device: modes 1 and 2 take their MTTKRP from the shared contraction
     T = X_(0)^T A_0 (csrc/pairnode.cuh), so an iteration runs two tensor-sized contractions instead of three. */
  double pair_gemm_ms;       /* timing: CUDA-event time summed over the T contractions (part of mttkrp_ms) */
  double pair_leaf_ms;       /* timing: CUDA-event time summed over the leaf kernels that read T (part of mttkrp_ms) */
  double tensor_flops;       /* flop that actually ran on the FP64 tensor cores (== mttkrp_flops without the pair node) */
  int32_t tree;              /* 1 when the pair node was used by this run */
  int32_t fused_leaf_blocks; /* > 0: the first leaf of the 3-mode pair node rode in the contraction's epilogue; the number
                                of partial results per element that pair_partial_reduce_kernel summed (ceil(I2 / tile)) */
  int32_t sweep_period;      /* 2: the multi-sweep dimension tree ran (3 modes: the contraction over mode 1 also serves
                                mode 0 of the next iteration, three tensor-sized contractions per two iterations);
                                1: every iteration runs the same contractions */
} cals_b200_report;

typedef struct cals_b200_model_stats {
  uint64_t iters;    /* Ktensor::iters */
  double error;      /* Ktensor::approx_error */
  double fit;        /* Ktensor::fit */
  double old_fit;    /* Ktensor::old_fit */
  int32_t chol_info; /* number of Cholesky failures met (reference only logs dpotrf's info, update.cpp:184) */
} cals_b200_model_stats;

/* ---- lifetime ------------------------------------------------------------------------------------------------ */
int cals_b200_create(cals_b200_ctx **ctx, int device);
int cals_b200_destroy(cals_b200_ctx *ctx);
const char *cals_b200_last_error(const cals_b200_ctx *ctx); /* ctx may be NULL: last error of create() */

/* ---- target tensor  (replaces X.allocate_cudata + send_to_device_async, reference src/cals.cpp:142-147) ------- */
/* Uploads X (prod(modes) doubles, mode 0 fastest), builds the device layouts the kernels read, and computes
 * ||X|| (Tensor::norm, include/tensor.h:196) on the device.  The call only ENQUEUES that work on the context's stream
 * (so that queueing the models on the host overlaps with it): host_X must stay valid and unchanged until the next
 * call that synchronises (cals_b200_run, cals_b200_tensor_norm, cals_b200_jk_norms, cals_b200_mttkrp). */
int cals_b200_set_tensor(cals_b200_ctx *ctx, int n_modes, const uint64_t *modes, const double *host_X);
/* Same with X already in device memory (dense, unpadded). */
int cals_b200_set_tensor_dev(cals_b200_ctx *ctx, int n_modes, const uint64_t *modes, const double *X_dev);

/* ---- tensor sliced along one mode over several GPUs (BASELINE config 5; no reference counterpart) ------------- */
/* Every GPU holds the slab [cuts[rank], cuts[rank+1]) of mode `slice_mode` (host_slab: dense, same layout as X with
 * that extent along slice_mode) and ALL factor columns; every MTTKRP is followed by an exchange over NVLink peer
 * memory (partial sums added in rank order on every GPU, row blocks gathered for the sliced mode), after which the
 * per-model updates run replicated and bit-identical on all GPUs.  Call order on every rank:
 *   cals_b200_comm_alloc -> exchange handles / pointers between ranks -> cals_b200_comm_connect ->
 *   cals_b200_set_tensor_slab -> combine the local norms: cals_b200_tensor_norm / cals_b200_set_tensor_norm ->
 *   configure / enqueue the SAME models on every rank / run / fetch (every rank holds all results).
 * `modes` are the extents of the whole tensor; cuts has world+1 entries, inner cuts even. */
int cals_b200_comm_alloc(cals_b200_ctx *ctx, int rank, int world, uint64_t capacity_doubles,
                         void *ipc_handle_out /* 64 bytes (cudaIpcMemHandle_t) or NULL */);
/* capacity_doubles >= max_n(I_n rounded up to even) * buffer_cols. */
int cals_b200_comm_local_block(cals_b200_ctx *ctx, void **block_dev_out);
/* One process per GPU: ipc_handles = world x 64 bytes in rank order (own entry ignored), the other two NULL.
 * One process driving all GPUs: ipc_handles NULL, peer_blocks_dev[r] = cals_b200_comm_local_block of rank r,
 * peer_devices[r] = its CUDA ordinal. */
int cals_b200_comm_connect(cals_b200_ctx *ctx, const void *ipc_handles, void *const *peer_blocks_dev,
                           const int *peer_devices);
/* Unmap the peers' exchange blocks (own block stays).  Every rank calls this, then synchronises with the others,
 * BEFORE any rank frees its block (cals_b200_comm_alloc again, or cals_b200_destroy): CUDA IPC does not allow the
 * exporter to free memory that an importer still has mapped. */
int cals_b200_comm_disconnect(cals_b200_ctx *ctx);
int cals_b200_set_tensor_slab(cals_b200_ctx *ctx, int n_modes, const uint64_t *modes, int slice_mode,
                              const uint64_t *cuts, const double *host_slab);
/* After set_tensor_slab, cals_b200_tensor_norm returns the norm of the local slab; the caller combines
 * sqrt(sum_r norm_r^2) and installs it with this call (Tensor::norm of the whole tensor). */
int cals_b200_set_tensor_norm(cals_b200_ctx *ctx, double norm);

/* ---- parameters (CalsParams, reference include/cals.h:138-159) ------------------------------------------------ */
int cals_b200_configure(cals_b200_ctx *ctx, uint64_t buffer_cols, uint64_t max_iterations, double tol,
                        unsigned flags);
/* CalsParams::line_search / line_search_method / line_search_interval / line_search_step (reference include/cals.h:
 * 153-156, src/utils/line_search.cpp).  method 0 = NO_ERROR_CHECKING, 1 = ERROR_CHECKING_SERIAL; step 0 = cbrt of the
 * model's iteration count (src/cals.cpp:317-318); interval >= 2.  Off by default, as in the reference. */
int cals_b200_set_line_search(cals_b200_ctx *ctx, int enabled, int method, int interval, double step);
/* CalsReport::ls_performed / ls_failed of the last run (reference include/cals.h:52-53). */
int cals_b200_line_search_counts(cals_b200_ctx *ctx, uint64_t *performed, uint64_t *failed);
/* 0: no per-kernel timing (default).  1: bracket MTTKRP / update kernels with CUDA events (adds syncs at the end). */
int cals_b200_set_timing(cals_b200_ctx *ctx, int level);
int cals_b200_set_mttkrp_variant(cals_b200_ctx *ctx, int variant);
/* CalsParams::mttkrp_method (reference include/cals.h:148, mttkrp::MTTKRP_METHOD in include/utils/mttkrp.h): 1 (default,
 * AUTO / TWOSTEP0 / TWOSTEP1) lets a 3-mode tensor held whole by one device take the MTTKRPs of modes 1 and 2 from
 * the shared contraction T = X_(0)^T A_0 (csrc/pairnode.cuh); 0 (method MTTKRP) runs one full MTTKRP per mode. */
int cals_b200_set_pair_node(cals_b200_ctx *ctx, int enabled);

/* ---- model queue (KtensorQueue, reference include/cals.h:22; MultiKtensor::add, src/multi_ktensor.cpp:41) ----- */
int cals_b200_clear_models(cals_b200_ctx *ctx);
/* host_factors[n] -> I_n x rank column-major (ld = I_n).  jk_mode < 0: regular model; else the model is a
 * jackknife model with row jk_fiber of factor jk_mode forced to zero (Ktensor::to_jk, include/ktensor.h:276). */
int cals_b200_enqueue_model(cals_b200_ctx *ctx, uint64_t rank, const double *const *host_factors, int jk_mode,
                            int64_t jk_fiber, int *model_id);

/* The same for a whole queue in one call: host_factors[m * n_modes + n]; jk_modes / jk_fibers may be NULL (no
 * jackknife models).  Model ids are the queue positions. */
int cals_b200_enqueue_models(cals_b200_ctx *ctx, uint64_t n_models, const uint64_t *ranks,
                             const double *const *host_factors, const int *jk_modes, const int64_t *jk_fibers);

/* ---- the hot path: the do/while loop of cals::cp_cals (reference src/cals.cpp:174-382) ------------------------- */
/* Uploads the queued models, runs concurrent ALS until every model has been evicted, leaves results on the device. */
int cals_b200_run(cals_b200_ctx *ctx, cals_b200_report *report);
/* Re-runs from the initial factors that are already resident on the device (no host->device traffic). */
int cals_b200_rerun(cals_b200_ctx *ctx, cals_b200_report *report);

/* ---- results (Ktensor::detach copies the result back, reference src/ktensor.cpp:127-135) ----------------------- */
int cals_b200_fetch_model(cals_b200_ctx *ctx, int model_id, double *const *factors_out, double *lambda_out,
                          cals_b200_model_stats *stats);
/* All models at once: factors_out[model*n_modes + n]; lambda_out[model]; stats[model]. Any pointer may be NULL. */
int cals_b200_fetch_all(cals_b200_ctx *ctx, double *const *factors_out, double *const *lambda_out,
                        cals_b200_model_stats *stats);

/* ---- core consistency (CORCONDIA, Bro & Kiers, J. Chemometrics 17 (2003) 274-286; extension, no reference
 * counterpart) ---------------------------------------------------------------------------------------------------- */
/* The core consistency diagnostic of every queued model, computed on the device: CC = 100 (1 - sum (G - I)^2 / R) with G
 * the least-squares Tucker core of X for the model's factors (A_0 = F_0 diag(lambda), A_n = F_n) and I the superdiagonal
 * identity.  After cals_b200_run / cals_b200_rerun the fitted factors and lambda are used; before any run (or after
 * the queue changed) the enqueued factors with lambda = 1.  A jackknife model leaves out its row of mode 0.
 * cc_out and status_out (may be NULL) get one entry per queued model, in model-id order; status 0 = computed,
 * 1 = rank above the limit (96 for 3 modes, 64 for 4), 2 = some A_n^T A_n is not numerically positive definite (rank
 * above an extent, equal columns, lambda = 0); cc is NaN unless the status is 0.  Tensors of 3 and 4 modes held whole by
 * this device only.  Nothing that a later fetch, run or rerun returns changes. */
int cals_b200_core_consistency(cals_b200_ctx *ctx, double *cc_out, int32_t *status_out);

/* ---- NNLS active sets (Ktensor::active_set, reference include/ktensor.h:36; they persist across calls there) ---- */
/* active[n] / active_out[n] -> I_n x rank bytes, row-major (byte [row * rank + col]); 1 = the entry is constrained
 * to zero.  Models start with every constraint active unless set here after enqueueing; fetch after a run. */
int cals_b200_set_model_active_set(cals_b200_ctx *ctx, int model_id, const uint8_t *const *active);
int cals_b200_fetch_model_active_set(cals_b200_ctx *ctx, int model_id, uint8_t *const *active_out);

/* ---- single-operation hooks (parity tests against the oracle; also the reference's unit seams) ----------------- */
int cals_b200_tensor_norm(cals_b200_ctx *ctx, double *norm_out);
/* utils::calculate_jackknifing_norms (reference src/utils/utils.cpp:103-152): out has modes[0] entries. */
int cals_b200_jk_norms(cals_b200_ctx *ctx, double *out);
/* mttkrp::mttkrp (reference src/utils/mttkrp.cpp:562) over `cols` concatenated columns: host_factors[k] is
 * I_k x cols (entry `mode` is ignored), host_G receives I_mode x cols.  *ms_out (may be NULL) = device time. */
int cals_b200_mttkrp(cals_b200_ctx *ctx, int mode, uint64_t cols, const double *const *host_factors, double *host_G,
                     int variant, int repeats, double *ms_out);

/* mttkrp::khatri_rao(A, B, workspace, params) (reference include/utils/mttkrp.h:88-89, src/utils/mttkrp.cpp:78-103; CUDA
 * twin khatri_rao_cuda, src/utils/khatri_rao.cu:40): K[ib + rows_B * ia, c] = A[ia, c] * B[ib, c] for `cols` columns,
 * all matrices column-major and dense (ld = rows).  The iteration path never materialises this product; the hook
 * exists for callers of that API function. */
int cals_b200_khatri_rao(cals_b200_ctx *ctx, const double *host_A, uint64_t rows_A, const double *host_B,
                         uint64_t rows_B, uint64_t cols, double *host_K);

/* CalsReport::cols (reference include/cals.h:62, filled at src/cals.cpp:214): the number of active multi-factor
 * columns in every global iteration of the last run.  Writes min(*n_out, capacity) entries; *n_out = iterations
 * logged (the device keeps the first 65536). */
int cals_b200_fetch_iteration_cols(cals_b200_ctx *ctx, uint32_t *cols_out, uint64_t capacity, uint64_t *n_out);

/* ---- page-locked host memory for the caller's tensors (so that set_tensor / enqueue run at full link speed) ------ */
/* Returns NULL when there is no CUDA device (callers then use ordinary memory); free with cals_b200_host_free. */
void *cals_b200_host_alloc(size_t bytes);
void cals_b200_host_free(void *p);

/* ---- introspection --------------------------------------------------------------------------------------------- */
/* The CUDA stream (cudaStream_t) every kernel and copy of this context is issued on, so that a caller can record its
 * own CUDA events around calls (bench.py times the steps with events on this stream). */
int cals_b200_stream(cals_b200_ctx *ctx, void **stream_out);
int cals_b200_device_info(cals_b200_ctx *ctx, int *sm_count, size_t *free_bytes, size_t *total_bytes);
const char *cals_b200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* CALS_B200_H */
