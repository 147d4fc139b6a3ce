// Device-side model queue: the MultiKtensor bookkeeping of the reference without host round trips.
//
//   admission  : FIFO, stop at the first model that does not fit           reference src/cals.cpp:182-192,
//                (first-fit == append, because the buffer is compacted)    src/multi_ktensor.cpp:14-39,41-130
//   eviction   : copy the model's columns back to its own ("home") storage reference src/multi_ktensor.cpp:132-163,
//                                                                           src/ktensor.cpp:127-135
//   compaction : stable shift of the live models to the left               reference src/multi_ktensor.cpp:188-264
//
// Compaction is a gather from the old buffer into the other one of a ping-pong pair (in-place overlapping shifts would
// need a grid-wide ordering); newly admitted models are gathered from their home columns in the same pass.
#pragma once
#include <cuda_runtime.h>

#include "common.cuh"
#include "mttkrp.cuh"

namespace calsb200 {

struct SchedParams {
  SchedState *st;
  ModelDesc *models;
  int *live;       // [max_live] model ids in column order (current)
  int *live_tmp;   // scratch
  int *gather_src; // [buffer_cols] new column j <- (>=0: old buffer column, <0: home column -1-src)
  int *evict_dst;  // [buffer_cols] old column j -> home column, or -1
  int *host_flags; // mapped pinned host memory: [0] done, [1] global_iter (low 31 bits), [2] n_live
  PlanArgs plans;  // MTTKRP work partition per mode, rebuilt whenever the live column count changes
  unsigned *iter_cols; // [ITER_LOG_CAP] active column count of every executed iteration (CalsReport::cols)
  int contractions;    // tensor-sized contractions of this pass (not counting the fallback MTTKRP below)
  int carry;           // odd pass of the multi-sweep schedule: mode 0 takes the carried T, or its own MTTKRP when the
                       // columns change in this pass (SchedState::carry_ok)
};
constexpr int ITER_LOG_CAP = 65536;

// One warp.  Lane 0 does the eviction / compaction bookkeeping (the live list is short and this part only runs when a
// model was flagged); admission -- up to hundreds of models and thousands of columns in the first iteration of a run --
// is done by the whole warp: 32 queued models at a time, a warp scan of their ranks decides how many still fit, every
// lane fills the gather list of its own model.  Then one thread per mode rebuilds that mode's MTTKRP plan if the column
// count changed.
__global__ void __launch_bounds__(32) sched_kernel(const SchedParams p) {
  pdl_enter();
  SchedState *st = p.st;
  const int lane = threadIdx.x;
  __shared__ int sh_col, sh_nlive, sh_changed, sh_done, sh_C_before;

  if (lane == 0) {
    sh_done = st->done;
    sh_C_before = st->C;
    if (st->done) {
      st->changed = 0;
      st->carry_ok = 0;
    } else {
      const int B = st->buffer_cols;
      bool changed = false;
      // always_evict_first: evict the leftmost live model, whatever its state (reference src/cals.cpp:348-354)
      if ((st->flags & 2u) && st->global_iter > 0 && st->n_live > 0) {
        p.models[p.live[0]].state = MODEL_EVICT;
        st->n_evict = 1;
      }
      int n_live = st->n_live, col = 0, kept = 0;
      if (st->n_evict > 0) {
        for (int j = 0; j < B; j++)
          p.evict_dst[j] = -1;
        for (int li = 0; li < n_live; li++) {
          const int m = p.live[li];
          ModelDesc &md = p.models[m];
          if (md.state == MODEL_EVICT) {
            for (int j = 0; j < md.rank; j++)
              p.evict_dst[md.col + j] = md.home_col + j;
            md.state = MODEL_DONE;
          } else {
            for (int j = 0; j < md.rank; j++)
              p.gather_src[col + j] = md.col + j;
            md.col = col;
            col += md.rank;
            p.live_tmp[kept++] = m;
          }
        }
        for (int li = 0; li < kept; li++)
          p.live[li] = p.live_tmp[li];
        n_live = kept;
        changed = true;
        st->n_evict = 0;
      } else {
        col = st->C;
      }
      sh_col = col;
      sh_nlive = n_live;
      sh_changed = changed ? 1 : 0;
    }
  }
  __syncwarp();
  if (sh_done)
    return;

  // ---- admission: FIFO, stop at the first model that does not fit (reference src/cals.cpp:182-192; first-fit equals
  // append because the buffer is compact, src/multi_ktensor.cpp:14-39) ----
  {
    const int B = st->buffer_cols, n_models = st->n_models;
    int next = st->next, col = sh_col, n_live = sh_nlive;
    bool changed = sh_changed != 0, admitted_any = false;
    unsigned long long comp = 0;
    const int next0 = next;
    for (bool more = true; more && next < n_models;) {
      const int m = next + lane;
      const int rank = m < n_models ? p.models[m].rank : 0x3fffffff; // beyond the queue: never fits
      int incl = rank > B ? B + 1 : rank;                             // clamp: sums stay far from overflow
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o)
          incl = min(incl + v, B + 1);
      }
      const bool fits = col + incl <= B; // monotone in the lane index
      const unsigned mask = __ballot_sync(0xffffffffu, fits);
      const int n_fit = __popc(mask);
      if (n_fit > 0 && !changed && !admitted_any) {
        // first structural change of this iteration without evictions: identity map for the resident columns
        for (int j = lane; j < B; j += 32)
          p.evict_dst[j] = -1;
        for (int j = lane; j < col; j += 32)
          p.gather_src[j] = j;
      }
      if (fits) {
        ModelDesc &md = p.models[m];
        const int my_col = col + incl - rank;
        for (int j = 0; j < rank; j++)
          p.gather_src[my_col + j] = -1 - (md.home_col + j);
        md.col = my_col;
        md.state = MODEL_LIVE;
        md.iters = 1; // reference src/multi_ktensor.cpp:96
        p.live[n_live + lane] = m;
      }
      if (n_fit > 0) {
        admitted_any = true;
        const int total = __shfl_sync(0xffffffffu, incl, n_fit - 1);
        comp += (unsigned long long)total;
        col += total;
        n_live += n_fit;
        next += n_fit;
      }
      more = (n_fit == 32);
    }
    __syncwarp();
    if (lane == 0) {
      changed = changed || admitted_any;
      st->next = next;
      st->n_admitted += (unsigned long long)(next - next0);
      st->comp_sum += comp;
      st->n_live = n_live;
      st->C = col;
      st->changed = changed ? 1 : 0;
      if (changed)
        st->cur ^= 1;
      const bool carry_ok = p.carry && !changed; // a moved column or a flipped buffer no longer matches the carried T
      st->carry_ok = carry_ok ? 1 : 0;
      if (n_live == 0 && next >= n_models) {
        st->done = 1;
      } else {
        if (st->global_iter < (unsigned long long)ITER_LOG_CAP)
          p.iter_cols[st->global_iter] = (unsigned)col;
        st->global_iter += 1; // reference: rep.iter counts executed loop bodies (src/cals.cpp:175-176)
        st->col_iter_sum += (unsigned long long)col;
        st->contraction_cols += (unsigned long long)col * (unsigned)(p.contractions + (p.carry && !carry_ok ? 1 : 0));
      }
      p.host_flags[1] = (int)(st->global_iter & 0x7fffffff);
      p.host_flags[2] = n_live;
      __threadfence_system();
      p.host_flags[0] = st->done;
      sh_col = col;
    }
  }
  __syncwarp();
  // A plan depends on the column count only, so it survives from run to run: a re-run with the same queue (every
  // benchmark step, every call of a parameter sweep) finds its tables in place instead of spending ~0.1 ms of a single
  // thread per mode on rebuilding them.
  const int C_now = sh_col;
  const int tail = st->narrow_on ? narrow_cols(C_now) : 0; // columns left to the narrow instances (mttkrp.cuh)
  if (lane == 0)
    st->C_main = C_now - tail;
  if (C_now > 0 && lane < p.plans.n_modes) {
    if (p.plans.built_for[lane] != C_now - tail) {
      mttkrp_make_plan(p.plans.plan[lane], p.plans.shape[lane], C_now - tail, p.plans.G);
      p.plans.built_for[lane] = C_now - tail;
    }
    if (tail > 0 && p.plans.plan_narrow[lane] != nullptr && p.plans.built_for[CALS_MAX_MODES + lane] != tail) {
      mttkrp_make_plan(p.plans.plan_narrow[lane], p.plans.shape[lane], tail, p.plans.G);
      p.plans.built_for[CALS_MAX_MODES + lane] = tail;
    }
  }
}

// Column mover.  grid = (ceil(buffer_cols / COLS_PER_CTA), n_modes, 2): z == 0 copies evicted columns old buffer ->
// home, z == 1 gathers the new buffer from (old buffer | home).
constexpr int MOVE_COLS = 4;
__global__ void __launch_bounds__(256)
move_kernel(const Geom geo, const FactorPtrs fac, const SchedState *__restrict__ st,
            const int *__restrict__ gather_src, const int *__restrict__ evict_dst) {
  pdl_enter();
  if (!st->changed)
    return;
  const int n = blockIdx.y;
  const int rows = geo.dims[n], ld = geo.ldF[n];
  const int cur = st->cur; // already flipped by the scheduler: cur is the NEW buffer
  const double *oldb = fac.buf[cur ^ 1][n];
  double *newb = fac.buf[cur][n];
  double *home = fac.home[n];
  const int j0 = blockIdx.x * MOVE_COLS;
  if (blockIdx.z == 0) {
    for (int jj = 0; jj < MOVE_COLS; jj++) {
      const int j = j0 + jj;
      if (j >= st->buffer_cols)
        break;
      const int dst = evict_dst[j];
      if (dst < 0)
        continue;
      for (int r = threadIdx.x; r < rows; r += blockDim.x)
        home[(size_t)dst * ld + r] = oldb[(size_t)j * ld + r];
    }
  } else {
    for (int jj = 0; jj < MOVE_COLS; jj++) {
      const int j = j0 + jj;
      if (j >= st->C)
        break;
      const int src = gather_src[j];
      const double *s = src >= 0 ? oldb + (size_t)src * ld : home + (size_t)(-1 - src) * ld;
      for (int r = threadIdx.x; r < rows; r += blockDim.x)
        newb[(size_t)j * ld + r] = s[r];
    }
  }
}

} // namespace calsb200
