// Shared device/host structures of the B200 CP-CALS engine.
//
// Device-resident state replaces the reference's host-side MultiKtensor registry (include/multi_ktensor.h:12-47):
// every queued model owns a ModelDesc; the scheduler kernel (sched.cuh) admits / evicts / compacts without a host
// round trip and every compute kernel reads the live set from SchedState.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#define CALS_MAX_MODES 8
#define CALS_MAX_OUTER (CALS_MAX_MODES - 2)

enum ModelState : int { MODEL_QUEUED = 0, MODEL_LIVE = 1, MODEL_EVICT = 2, MODEL_DONE = 3 };

// One CP model (reference: Ktensor + RegistryEntry).  Factors of a queued / finished model live in the per-mode
// "home" matrices at columns [home_col, home_col+rank); while live they occupy buffer columns [col, col+rank).
struct ModelDesc {
  int rank;
  int home_col;
  int jk_mode; // -1: regular
  int jk_fiber;
  long long gram_off; // doubles; n_modes matrices of rank*rank, mode-major
  long long act_off;  // bytes into the active-set pool (NNLS): per mode an I_n x rank block, row-major
  int state;
  int col;
  int iters;
  int chol_info;
  double error, fit, old_fit;
  // line search (RegistryEntry::ls_params of the reference, include/multi_ktensor.h:20, include/utils/line_search.h:15-34)
  int ls_iter;         // iterations since the last extrapolation
  int ls_updated_last; // NO_ERROR_CHECKING: the previous iteration extrapolated
  int ls_trial;        // ERROR_CHECKING: a trial model of this iteration waits for its explicit error
  int b_iters;         // backup_ktensor: scalars (its factors / lambda live in the ls_backup matrices)
  double b_error, b_fit, b_old_fit;
};

struct SchedState {
  int n_models;
  int next;   // queue head (FIFO)
  int n_live;
  int C;      // active buffer columns
  int cur;    // which of the two factor buffers is current
  int changed; // set by the scheduler when columns have to move this iteration
  int done;
  int flags;  // CALS_B200_FORCE_MAX_ITER | CALS_B200_ALWAYS_EVICT_FIRST
  int max_iter;
  int buffer_cols;
  int n_evict; // models flagged for eviction by the last fit step
  int comm_error; // set by the exchange kernel when a peer GPU never arrived (slab mode)
  double tol;
  double x_norm;
  unsigned long long global_iter;
  unsigned long long n_admitted;
  unsigned long long comp_sum;
  unsigned long long col_iter_sum; // sum over executed iterations of the active column count C
  // line search (CalsParams::line_search*, reference include/cals.h:153-156)
  int ls_enabled, ls_method, ls_interval, ls_pad_;
  double ls_step; // 0: cbrt(model iteration), reference src/cals.cpp:317-318
  unsigned long long ls_performed, ls_failed;
  // Narrow column tail (mttkrp.cuh: narrow_cols): the contraction kernels' main instances work on columns [0, C_main),
  // their narrow instances on [C_main, C).  C_main == C unless narrow_on and the tail qualifies.
  int C_main;
  int narrow_on; // set by the host per run
  // Multi-sweep dimension tree (engine.cu: run_loop): an even pass leaves T = X x_1 A_1 behind for the mode-0 update of
  // the next pass.  carry_ok: this pass is odd and the scheduler moved no column, so that T still matches the buffer;
  // otherwise mode 0 runs its own MTTKRP.
  int carry_ok;
  int carry_pad_;
  unsigned long long contraction_cols; // sum over executed passes of C x the tensor-sized contractions the pass ran
};

// eviction predicate + iteration counter (reference src/cals.cpp:336-347); called by exactly one thread per model
__device__ __forceinline__ void decide_eviction(ModelDesc &md, SchedState *st) {
  if (st->flags & 2u) // always_evict_first: the scheduler evicts the leftmost model
    return;
  const int iters = md.iters;
  bool evict;
  if (st->flags & 1u)
    evict = iters >= st->max_iter;
  else
    evict = (fabs(md.old_fit - md.fit) < st->tol) || (iters >= st->max_iter);
  if (evict) {
    md.state = MODEL_EVICT;
    atomicAdd(&st->n_evict, 1);
  } else
    md.iters = iters + 1;
}

// Programmatic dependent launch (sm_90+): the kernels of one CALS iteration form a chain; each is launched with
// cudaLaunchAttributeProgrammaticStreamSerialization so that its CTAs are scheduled -- block start-up, parameter and
// descriptor fetch, the first instruction lines -- while its predecessor is still draining, and blocks here until the
// predecessor has completed and its writes are visible.  Every thread of every kernel of the chain calls pdl_wait()
// before it touches anything another kernel writes (no early return in front of it: a grid that completed without
// waiting would let ITS successor run ahead of a still-running grand-predecessor).  Without the launch attribute both
// instructions are no-ops.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_enter() {
  pdl_wait();
  pdl_trigger();
}

// Geometry shared by all kernels: extents and leading dimensions.
struct Geom {
  int n_modes;
  int dims[CALS_MAX_MODES];
  int ldF[CALS_MAX_MODES]; // leading dimension of factor buffers / home matrices / G (dims rounded up to even)
};

struct FactorPtrs {
  double *buf[2][CALS_MAX_MODES]; // ping-pong multi-factor buffers, ldF[n] x buffer_cols
  double *home[CALS_MAX_MODES];   // ldF[n] x total_cols
};

static inline int round_up_int(int x, int m) { return (x + m - 1) / m * m; }
