// Line search (reference src/utils/line_search.cpp, driven from src/cals.cpp:203-212 and :309-333), per live model and
// entirely on the device: every `interval` iterations a model is extrapolated along (current - snapshot),
//   NO_ERROR_CHECKING      blindly; the next iteration compares errors and returns to a backup if it got worse,
//   ERROR_CHECKING_SERIAL  as a trial model whose explicit error ||X - M|| decides whether it replaces the model.
// One CTA per live model (they are independent).  Snapshots ("prev_ktensor"), backups and trial models live in
// matrices shaped like the home matrices (pitch ldF, a model's columns at home_col).
#pragma once
#include <cuda_runtime.h>

#include "common.cuh"
#include "update.cuh"

namespace calsb200 {

struct LsParams {
  Geom geo;
  FactorPtrs fac;
  double *prev[CALS_MAX_MODES];   // snapshot; doubles as the trial model under ERROR_CHECKING
  double *backup[CALS_MAX_MODES]; // NO_ERROR_CHECKING only
  double *prev_lambda, *backup_lambda, *lambda_home;
  double *gram_pool;
  ModelDesc *models;
  const int *live;
  SchedState *st;
  const double *X; // caller-order device copy of the tensor (pitch ldX0)
  int ldX0;
  long long rest0;  // number of mode-0 fibres
  double *partial;  // [max_live][chunks] partial sums of squares of X - trial model
  int chunks;
};

// Ktensor::copy of the factors (reference src/ktensor.cpp:162-179): buffer columns <-> home-indexed matrices
__device__ __forceinline__ void ls_copy(double *dst, const double *src, int rows, int ld, int R) {
  for (int e = threadIdx.x; e < rows * R; e += blockDim.x) {
    const int r = e % rows, c = e / rows;
    dst[(size_t)c * ld + r] = src[(size_t)c * ld + r];
  }
}

// ops::update_gramians (reference src/utils/utils.cpp:174-185) from factors in global memory
__device__ void ls_gramians(const LsParams &p, const ModelDesc &md, double *const *F) {
  const int R = md.rank;
  double *grams = p.gram_pool + md.gram_off;
  for (int n = 0; n < p.geo.n_modes; n++) {
    const int rows = p.geo.dims[n], ld = p.geo.ldF[n];
    for (int e = threadIdx.x; e < R * R; e += blockDim.x) {
      const int i = e % R, j = e / R;
      const double *ci = F[n] + (size_t)i * ld, *cj = F[n] + (size_t)j * ld;
      double g = 0.0;
      for (int r = 0; r < rows; r++)
        g += ci[r] * cj[r];
      grams[(size_t)n * R * R + e] = g;
    }
  }
}

// Ktensor::normalize() (reference src/ktensor.cpp:85-99): unit 2-norm columns in every mode, lambda = product of norms.
// lambda must hold 1.0 on entry.  Warp per column.
__device__ void ls_normalize_all(const LsParams &p, int R, double *const *F, double *lambda) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int n = 0; n < p.geo.n_modes; n++) {
    const int rows = p.geo.dims[n], ld = p.geo.ldF[n];
    for (int c = warp; c < R; c += nw) {
      double *col = F[n] + (size_t)c * ld;
      double ss = 0.0;
      for (int r = lane; r < rows; r += 32)
        ss += col[r] * col[r];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1)
        ss += __shfl_xor_sync(0xffffffffu, ss, o);
      const double nrm = sqrt(ss), inv = 1.0 / nrm;
      for (int r = lane; r < rows; r += 32)
        col[r] *= inv;
      if (lane == 0)
        lambda[c] *= nrm;
    }
    __syncthreads(); // lambda[c] is updated by a different warp in the next mode only after this one is done
  }
}

// "Is it time to remember the model as it is now?" (reference src/cals.cpp:203-212) -- before the modes loop.
__global__ void __launch_bounds__(256) ls_snapshot_kernel(const LsParams p) {
  SchedState *st = p.st;
  if ((int)blockIdx.x >= st->n_live || !st->ls_enabled)
    return;
  const ModelDesc &md = p.models[p.live[blockIdx.x]];
  if (md.ls_iter != st->ls_interval - 1)
    return;
  const int cur = st->cur, R = md.rank;
  for (int n = 0; n < p.geo.n_modes; n++)
    ls_copy(p.prev[n] + (size_t)md.home_col * p.geo.ldF[n], p.fac.buf[cur][n] + (size_t)md.col * p.geo.ldF[n],
            p.geo.dims[n], p.geo.ldF[n], R);
  for (int c = threadIdx.x; c < R; c += blockDim.x)
    p.prev_lambda[md.home_col + c] = p.lambda_home[md.home_col + c];
}

// After the error/fit of the iteration: ls::line_search (reference src/utils/line_search.cpp:219-268) and, for
// NO_ERROR_CHECKING, the eviction decision that follows it.
__global__ void __launch_bounds__(256) ls_main_kernel(const LsParams p) {
  SchedState *st = p.st;
  if ((int)blockIdx.x >= st->n_live)
    return;
  ModelDesc &md = p.models[p.live[blockIdx.x]];
  const int cur = st->cur, R = md.rank, N = p.geo.n_modes, tid = threadIdx.x;
  const int method = st->ls_method, interval = st->ls_interval;
  double *F[CALS_MAX_MODES], *P[CALS_MAX_MODES], *B[CALS_MAX_MODES];
  for (int n = 0; n < N; n++) {
    F[n] = p.fac.buf[cur][n] + (size_t)md.col * p.geo.ldF[n];
    P[n] = p.prev[n] + (size_t)md.home_col * p.geo.ldF[n];
    B[n] = p.backup[n] ? p.backup[n] + (size_t)md.home_col * p.geo.ldF[n] : nullptr;
  }
  double *lam = p.lambda_home + md.home_col, *plam = p.prev_lambda + md.home_col;
  double *blam = p.backup_lambda ? p.backup_lambda + md.home_col : nullptr;

  // all threads read the decision inputs before anyone writes
  const int iters = md.iters;
  int ls_iter = md.ls_iter;
  const int updated_last = md.ls_updated_last;
  const double error = md.error, b_error = md.b_error;
  __syncthreads();
  if (tid == 0)
    md.ls_trial = 0;

  const bool skipped = (method == 0 && iters >= st->max_iter); // no extrapolation right before an eviction
  if (!skipped) {
    const double step = st->ls_step == 0.0 ? cbrt((double)iters) : st->ls_step;
    ls_iter++;
    if (method == 0) {
      bool restore = false;
      if (updated_last && b_error < error) { // the extrapolation made it worse: return to the backup
        restore = true;
        ls_iter = 0;
        for (int n = 0; n < N; n++)
          ls_copy(F[n], B[n], p.geo.dims[n], p.geo.ldF[n], R);
        for (int c = tid; c < R; c += blockDim.x)
          lam[c] = blam[c];
        __syncthreads();
        ls_gramians(p, md, F);
        if (tid == 0) {
          md.error = md.b_error;
          md.fit = md.b_fit;
          md.old_fit = md.b_old_fit;
          md.iters = md.b_iters;
          atomicAdd(&st->ls_failed, 1ull);
        }
        __syncthreads();
      }
      if (tid == 0)
        md.ls_updated_last = 0;
      if (!restore && ls_iter == interval) {
        ls_iter = 0;
        // backup_ktensor.copy(ktensor)
        for (int n = 0; n < N; n++)
          ls_copy(B[n], F[n], p.geo.dims[n], p.geo.ldF[n], R);
        for (int c = tid; c < R; c += blockDim.x)
          blam[c] = lam[c];
        if (tid == 0) {
          md.b_error = md.error;
          md.b_fit = md.fit;
          md.b_old_fit = md.old_fit;
          md.b_iters = md.iters;
        }
        __syncthreads();
        // line_search_no_error_checking (reference :23-68): denormalize both, extrapolate, normalize()
        {
          const int rows = p.geo.dims[0], ld = p.geo.ldF[0];
          for (int e = tid; e < rows * R; e += blockDim.x) {
            const int r = e % rows, c = e / rows;
            F[0][(size_t)c * ld + r] *= lam[c];
            P[0][(size_t)c * ld + r] *= plam[c];
          }
        }
        __syncthreads();
        for (int n = 0; n < N; n++) {
          const int rows = p.geo.dims[n], ld = p.geo.ldF[n];
          for (int e = tid; e < rows * R; e += blockDim.x) {
            const size_t o = (size_t)(e / rows) * ld + e % rows;
            const double f = F[n][o];
            F[n][o] = f + step * (f - P[n][o]);
          }
        }
        for (int c = tid; c < R; c += blockDim.x)
          lam[c] = 1.0;
        __syncthreads();
        ls_normalize_all(p, R, F, lam);
        ls_gramians(p, md, F);
        if (tid == 0) {
          md.error = 1.7976931348623157e308;
          md.old_fit = md.fit;
          md.fit = 1.0 - 1.7976931348623157e308; // calculate_new_fit(1.0), reference :38-39
          md.ls_updated_last = 1;
          atomicAdd(&st->ls_performed, 1ull);
        }
      }
    } else if (ls_iter == interval) { // ERROR_CHECKING_SERIAL: build the trial model (reference :96-109)
      ls_iter = 0;
      for (int n = 0; n < N; n++) {
        const int rows = p.geo.dims[n], ld = p.geo.ldF[n];
        for (int e = tid; e < rows * R; e += blockDim.x) {
          const int r = e % rows, c = e / rows;
          const size_t o = (size_t)c * ld + r;
          const double f = F[n][o];
          double t = f + step * (f - P[n][o]);
          if (n == 0)
            t *= lam[c]; // compute_error starts with denormalize() (reference src/utils/error.cpp:13)
          P[n][o] = t;
        }
      }
      for (int c = tid; c < R; c += blockDim.x)
        plam[c] = 1.0; // the trial's lambda after denormalisation; normalize() in ls_decide_kernel rebuilds it
      if (tid == 0) {
        md.ls_trial = 1;
        atomicAdd(&st->ls_performed, 1ull);
      }
    }
  }
  __syncthreads();
  if (tid == 0) {
    md.ls_iter = ls_iter;
    if (method == 0)
      decide_eviction(md, st);
  }
}

// ||X - trial model||^2 of every model with a trial, by explicit reconstruction (error::compute_error, reference
// src/utils/error.cpp:7-31; any number of modes).  grid = (max_live, chunks): CTA (m, k) handles the k-th share of the
// mode-0 fibres and writes one partial sum; the partials are added in chunk order by ls_decide_kernel (deterministic).
__global__ void __launch_bounds__(256) ls_explicit_error_kernel(const LsParams p) {
  SchedState *st = p.st;
  if ((int)blockIdx.x >= st->n_live)
    return;
  const ModelDesc &md = p.models[p.live[blockIdx.x]];
  if (!md.ls_trial)
    return;
  extern __shared__ double lsm[]; // w[R] + 32
  double *w = lsm, *red = lsm + md.rank;
  const int R = md.rank, N = p.geo.n_modes, tid = threadIdx.x;
  const int I0 = p.geo.dims[0], ld0 = p.geo.ldF[0];
  const double *T0 = p.prev[0] + (size_t)md.home_col * ld0;
  const long long per = (p.rest0 + p.chunks - 1) / p.chunks;
  const long long o0 = per * blockIdx.y, o1 = min(p.rest0, o0 + per);
  double acc = 0.0;
  for (long long o = o0; o < o1; o++) {
    __syncthreads();
    for (int r = tid; r < R; r += blockDim.x) { // product of the slower modes' trial factors for component r
      long long rem = o;
      double v = 1.0;
      for (int n = 1; n < N; n++) {
        const int idx = (int)(rem % p.geo.dims[n]);
        rem /= p.geo.dims[n];
        v *= p.prev[n][(size_t)(md.home_col + r) * p.geo.ldF[n] + idx];
      }
      w[r] = v;
    }
    __syncthreads();
    const double *x = p.X + o * (long long)p.ldX0;
    for (int i = tid; i < I0; i += blockDim.x) {
      double m = 0.0;
      for (int r = 0; r < R; r++)
        m += w[r] * T0[(size_t)r * ld0 + i];
      const double d = x[i] - m;
      acc += d * d;
    }
  }
  acc = block_sum(acc, red);
  if (tid == 0)
    p.partial[(size_t)blockIdx.x * p.chunks + blockIdx.y] = acc;
}

// ERROR_CHECKING_SERIAL: accept or drop the trial (reference src/utils/line_search.cpp:111-150), then the eviction
// decision for every live model.
__global__ void __launch_bounds__(256) ls_decide_kernel(const LsParams p) {
  SchedState *st = p.st;
  if ((int)blockIdx.x >= st->n_live)
    return;
  ModelDesc &md = p.models[p.live[blockIdx.x]];
  const int cur = st->cur, R = md.rank, N = p.geo.n_modes, tid = threadIdx.x;
  if (md.ls_trial) {
    double e2 = 0.0;
    for (int k = 0; k < p.chunks; k++)
      e2 += p.partial[(size_t)blockIdx.x * p.chunks + k];
    const double e_new = sqrt(e2);
    const double e_old = md.error;
    __syncthreads();
    if (e_new < e_old) {
      double *F[CALS_MAX_MODES], *P[CALS_MAX_MODES];
      for (int n = 0; n < N; n++) {
        F[n] = p.fac.buf[cur][n] + (size_t)md.col * p.geo.ldF[n];
        P[n] = p.prev[n] + (size_t)md.home_col * p.geo.ldF[n];
      }
      // compute_error leaves the trial normalised (reference src/utils/error.cpp:28); its factors -- not its lambda --
      // replace the model's
      ls_normalize_all(p, R, P, p.prev_lambda + md.home_col);
      for (int n = 0; n < N; n++)
        ls_copy(F[n], P[n], p.geo.dims[n], p.geo.ldF[n], R);
      __syncthreads();
      ls_gramians(p, md, F);
      if (tid == 0) {
        md.error = e_new;
        md.old_fit = md.fit;
        md.fit = 1.0 - fabs(e_new) / st->x_norm;
      }
    } else if (tid == 0)
      atomicAdd(&st->ls_failed, 1ull);
    __syncthreads();
  }
  if (tid == 0) {
    md.ls_trial = 0;
    decide_eviction(md, st);
  }
}

} // namespace calsb200
