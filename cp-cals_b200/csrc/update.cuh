// Per-model small operations, one CTA per live model, fused into a single kernel per mode:
//
//   H = hadamard of the other modes' Gramians     ops::hadamard_but_one      reference src/utils/utils.cpp:161-172
//   L = chol_lower(H)                               dpotrf('L')                reference src/utils/update.cpp:183-185
//   F = G * L^-T * L^-1 (row-wise two solves)       2 x dtrsm                  reference src/utils/update.cpp:187-190
//   jackknife row := 0                              Ktensor::set_jk_fiber(0)   reference include/ktensor.h:316-325
//   lambda, column scaling                          Ktensor::normalize(n, it)  reference src/ktensor.cpp:66-83
//   Gram_n = F^T F                                  ops::update_gramian        reference src/utils/utils.cpp:174-178
// and, after the last mode,
//   P = hadamard of all Gramians, fast error, fit   ops::hadamard_all, error::compute_fast_error,
//                                                   Ktensor::calculate_new_fit reference src/utils/utils.cpp:156,
//                                                   src/utils/error.cpp:64-89, include/ktensor.h:178-183
//   eviction predicate / iters++                    reference src/cals.cpp:336-347
//
// The MTTKRP result G is read from its own buffer and the updated factor is written to the multi-factor buffer, so the
// last mode's G is still intact for the error term (the reference keeps a copy: G_last, src/cals.cpp:75,230-234).
#pragma once
#include <cuda_runtime.h>

#include "common.cuh"
#include "mttkrp.cuh"

namespace calsb200 {

constexpr int UPDATE_THREADS = 256;

struct UpdateParams {
  int mode;
  int n_modes;
  int rows;      // I_n
  int ld;        // ldF[n] == ldG
  int chunk_rows; // rows staged in shared memory at a time (multiple of 32)
  int chunk_pitch; // odd pitch (in doubles) of the staged chunk
  int max_rank;
  const double *G;         // MTTKRP result, ld x C
  double *F[2];            // multi-factor buffers for this mode
  double *gram_pool;
  double *lambda_home;     // per home column
  const double *x_norms_jk; // modes[0] entries or nullptr
  ModelDesc *models;
  const int *live;
  SchedState *st;
  // fused reduction of the stream-K partial tiles (replaces mttkrp_reduce_kernel on the iteration path): when
  // plan != nullptr the MTTKRP result is not read from G but summed here, per (m,n) pair in segment order, from the
  // partial-tile workspace the DMMA kernel has just written; for the last mode the sum is also written to G (the
  // error term needs it after the solve).
  const int *plan;
  const double *ws;
  int plan_ctas;  // gridDim.x of the DMMA kernel (layout of the plan tables)
  int tile_elems; // M_TILE * N_TILE of this mode's DMMA kernel
  int n_tile;     // N_TILE
  double *G_out;  // == G (mutable alias)
  // non-negative update (update_method == NNLS)
  int nnls;                 // 0: Cholesky solve, 1: row-wise active-set NNLS
  int nnls_warps;           // warps of the CTA that work on rows (each owns a scratch block in shared memory)
  int rows_before;          // sum of the extents of the modes below this one (offset into a model's active sets)
  unsigned char *act_pool;  // per model: for every mode an I_n x R block, row-major, 1 = constrained to zero
  int table_off;            // doubles from the start of shared memory to the tile lookup tables of the fused reduction
  long long *prof;          // tuning aid (CALS_B200_UPDATE_PROF=1): 16 clock64() stamps per CTA, nullptr otherwise
  // H, its Cholesky factor, the inverses of its diagonal blocks, 1 / diag(L) and diag(H) of every live model, computed
  // by prefactor_kernel while the kernel in front of this one was running (nullptr: computed here)
  const double *pref;
  long long pref_stride;    // doubles per live slot
};

struct PrefactorParams {
  int mode, n_modes;
  const double *gram_pool;
  const ModelDesc *models;
  const int *live;
  const SchedState *st;
  double *pref;
  long long pref_stride;
  int max_rank; // largest narrow rank: wide models (wide.cuh) are skipped
};
#define CALS_PROF(slot)                                                                                                \
  do {                                                                                                                 \
    if (p.prof != nullptr && threadIdx.x == 0)                                                                         \
      p.prof[(size_t)blockIdx.x * 16 + (slot)] = clock64();                                                            \
  } while (0)

__device__ __forceinline__ double block_sum(double v, double *scratch) {
  // scratch: >= 32 doubles of shared memory
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
    v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0)
    scratch[warp] = v;
  __syncthreads();
  double t = 0.0;
  if (warp == 0) {
    t = lane < (blockDim.x >> 5) ? scratch[lane] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
      t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0)
      scratch[0] = t;
  }
  __syncthreads();
  t = scratch[0];
  __syncthreads();
  return t;
}


// ------------------------------------------------------------------------------------------------------------------
// Row-wise active-set NNLS: update::update_factor_non_negative_constrained (reference src/utils/update.cpp:61-176),
// one warp per factor row, everything in shared memory.  Scratch per warp (doubles): y d w s sp [5R], Gp [R*R];
// ints: act [R], map [R+1].
struct NnlsScratch {
  double *y, *d, *w, *s, *sp, *Gp;
  int *act, *map;
};

__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
    v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int warp_sum_int(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
    v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Solve H_pp x = y_p for the passive set (dposv('L'), reference src/utils/update.cpp:18-46).  Returns the size of the
// passive set, or -1 when the Cholesky meets a non-positive pivot (CholFail).
__device__ int nnls_solve_passive(const double *H, int ldh, int R, const NnlsScratch &q, int lane) {
  __syncwarp();
  if (lane == 0) {
    int p = 0;
    for (int i = 0; i < R; i++)
      if (!q.act[i])
        q.map[p++] = i;
    q.map[R] = p;
  }
  __syncwarp();
  const int p = q.map[R];
  double *Gp = q.Gp, *sp = q.sp;
  for (int e = lane; e < p * p; e += 32) {
    const int a = e % p, b = e / p;
    Gp[a + b * p] = H[q.map[a] + q.map[b] * ldh];
  }
  for (int a = lane; a < p; a += 32)
    sp[a] = q.y[q.map[a]];
  __syncwarp();
  for (int j = 0; j < p; j++) {
    const double dj = Gp[j + j * p];
    if (!(dj > 0.0))
      return -1; // warp-uniform: every lane read the same value
    const double sd = sqrt(dj);
    __syncwarp();
    if (lane == 0)
      Gp[j + j * p] = sd;
    for (int i = j + 1 + lane; i < p; i += 32)
      Gp[i + j * p] /= sd;
    __syncwarp();
    const int t = p - j - 1;
    for (int e = lane; e < t * t; e += 32) {
      const int i = j + 1 + e % t, k = j + 1 + e / t;
      if (k <= i)
        Gp[i + k * p] -= Gp[i + j * p] * Gp[k + j * p];
    }
    __syncwarp();
  }
  for (int j = 0; j < p; j++) { // L z = y_p
    const double z = sp[j] / Gp[j + j * p];
    __syncwarp();
    if (lane == 0)
      sp[j] = z;
    for (int i = j + 1 + lane; i < p; i += 32)
      sp[i] -= Gp[i + j * p] * z;
    __syncwarp();
  }
  for (int j = p - 1; j >= 0; j--) { // L^T x = z
    const double x = sp[j] / Gp[j + j * p];
    __syncwarp();
    if (lane == 0)
      sp[j] = x;
    for (int i = lane; i < j; i += 32)
      sp[i] -= Gp[j + i * p] * x;
    __syncwarp();
  }
  return p;
}

__device__ __forceinline__ void nnls_scatter(double *dst, int R, int p, const NnlsScratch &q, int lane) {
  for (int i = lane; i < R; i += 32)
    dst[i] = 0.0;
  __syncwarp();
  for (int a = lane; a < p; a += 32)
    dst[q.map[a]] = q.sp[a];
  __syncwarp();
}
__device__ __forceinline__ double nnls_min_sp(int p, const NnlsScratch &q, int lane) {
  double m = 1.7976931348623157e308;
  for (int a = lane; a < p; a += 32)
    m = fmin(m, q.sp[a]);
  return warp_min(m);
}
__device__ __forceinline__ int nnls_count_passive(int R, const NnlsScratch &q, int lane) {
  int n = 0;
  for (int i = lane; i < R; i += 32)
    n += !q.act[i];
  return warp_sum_int(n);
}
__device__ __forceinline__ void nnls_multipliers(const double *H, int ldh, int R, const NnlsScratch &q, int lane) {
  for (int i = lane; i < R; i += 32) { // w = y - H d   (reference src/utils/update.cpp:49-57)
    double t = 0.0;
    for (int j = 0; j < R; j++)
      t += H[i + j * ldh] * q.d[j];
    q.w[i] = q.y[i] - t;
  }
  __syncwarp();
}

// One row: y = the row of the MTTKRP result in S (pitch `pitch`), result written back to S, active set updated in
// `arow` (global memory).  Returns 1 when a passive-block Cholesky failed inside the main loop or an iteration cap was
// hit (the reference has no caps; they only guard the GPU against a non-terminating corner case).
__device__ int nnls_row(const double *H, int ldh, int R, double tol, double *Srow, int pitch, unsigned char *arow,
                        const NnlsScratch &q, int lane) {
  int any = 0;
  for (int i = lane; i < R; i += 32) {
    const double yi = Srow[i * pitch];
    int a = arow[i];
    if (yi > 0.0)
      a = 0;
    q.y[i] = yi;
    q.d[i] = 0.0;
    q.act[i] = a;
    any |= !a;
  }
  any = __any_sync(0xffffffffu, any);
  __syncwarp();
  int p = 0;
  if (any) { // warm start from the previous active set (reference :88-117)
    p = nnls_solve_passive(H, ldh, R, q, lane);
    bool failed = p < 0;
    for (int guard = 0; !failed; guard++) {
      nnls_scatter(q.d, R, p, q, lane);
      if (!(nnls_min_sp(p, q, lane) <= tol))
        break;
      for (int i = lane; i < R; i += 32)
        if (q.d[i] <= tol) {
          q.d[i] = 0.0;
          q.act[i] = 1;
        }
      __syncwarp();
      if (nnls_count_passive(R, q, lane) == 0 || guard > 2 * R) {
        failed = true;
        break;
      }
      p = nnls_solve_passive(H, ldh, R, q, lane);
      failed = p < 0;
    }
    if (failed) {
      for (int i = lane; i < R; i += 32) {
        q.act[i] = 1;
        q.d[i] = 0.0;
      }
      __syncwarp();
    }
  }
  nnls_multipliers(H, ldh, R, q, lane);
  int trouble = 0;
  for (int outer = 0;; outer++) { // main loop (reference :122-170)
    double best = -1.7976931348623157e308;
    int bi = 0x7fffffff;
    for (int i = lane; i < R; i += 32)
      if (q.act[i] && q.w[i] > best) { // strictly greater: the first index of the maximum within this lane's sequence
        best = q.w[i];
        bi = i;
      }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ob > best || (ob == best && oi < bi)) {
        best = ob;
        bi = oi;
      }
    }
    if (bi == 0x7fffffff || !(best > tol))
      break;
    if (outer > 3 * R) {
      trouble = 1;
      break;
    }
    if (lane == 0)
      q.act[bi] = 0;
    p = nnls_solve_passive(H, ldh, R, q, lane);
    if (p < 0) {
      trouble = 1;
      break;
    }
    bool bad = false;
    for (int inner = 0; nnls_min_sp(p, q, lane) <= tol; inner++) { // inner loop (reference :131-155)
      nnls_scatter(q.s, R, p, q, lane);
      double alpha = 1.7976931348623157e308;
      for (int i = lane; i < R; i += 32)
        if (!q.act[i] && q.s[i] <= tol)
          alpha = fmin(alpha, q.d[i] / (q.d[i] - q.s[i]));
      alpha = warp_min(alpha);
      for (int i = lane; i < R; i += 32) {
        const double di = q.d[i] + alpha * (q.s[i] - q.d[i]);
        q.d[i] = di;
        if (fabs(di) < tol && !q.act[i]) {
          q.act[i] = 1;
          q.d[i] = 0.0;
        }
      }
      __syncwarp();
      if (nnls_count_passive(R, q, lane) == 0 || inner > 3 * R) {
        bad = true;
        break;
      }
      p = nnls_solve_passive(H, ldh, R, q, lane);
      if (p < 0) {
        bad = true;
        break;
      }
    }
    if (bad) {
      trouble = 1;
      break;
    }
    nnls_scatter(q.d, R, p, q, lane);
    nnls_multipliers(H, ldh, R, q, lane);
  }
  for (int i = lane; i < R; i += 32) {
    Srow[i * pitch] = q.d[i];
    arow[i] = (unsigned char)q.act[i];
  }
  __syncwarp();
  return trouble;
}

// ------------------------------------------------------------------------------------------------------------------
// Cholesky by ONE warp, in shared memory, while the other warps of the CTA stage the MTTKRP result.  Everything in this
// kernel is written as compact loops on purpose: it runs once per (model, mode), so a CTA executes every instruction
// only a few times and straight-line code runs at instruction-fetch speed (a fully unrolled register-resident
// factorisation was measured at 50 k cycles for R = 20; these loops take a fraction of that).
//
// H = L L^T, left-looking: for column j every lane owns one row i >= j and forms
//   s_i = H[i][j] - sum_{k<j} L[i][k] L[j][k]      (two running sums, loads only -- no store -> load chains)
// the diagonal s_j comes from lane 0 by shuffle, one reciprocal square root per column, L[i][j] = s_i * rinv.
// inv[j] = 1 / L[j][j].  The strict upper triangle of Hs keeps H.  Returns 1 when a pivot is not positive (dpotrf's
// info > 0; the reference only logs it and carries on, src/utils/update.cpp:183-185).
// The R x R matrices of this kernel (H / L, the diagonal-block inverses / the new Gramian) live in shared memory with
// leading dimension LD = R rounded up to 8 and zeros in the padding, so that the tensor-core loops below need no masks.
__device__ __forceinline__ int cholesky_warp(double *Hs, int LD, double *inv, int R, int lane) {
  int fail = 0;
  if (R <= 32) { // one row per lane, no pass loop
    const int i = lane;
    const double *li = Hs + i;
#pragma unroll 1
    for (int j = 0; j < R; j++) {
      const double *lj = Hs + j;
      double a0 = 0.0, a1 = 0.0;
      if (i >= j && i < R) {
        a0 = li[j * LD];
        int k = 0;
#pragma unroll 2
        for (; k + 2 <= j; k += 2) {
          a0 -= li[k * LD] * lj[k * LD];
          a1 -= li[(k + 1) * LD] * lj[(k + 1) * LD];
        }
        if (k < j)
          a0 -= li[k * LD] * lj[k * LD];
      }
      const double si = a0 + a1;
      const double d = __shfl_sync(0xffffffffu, si, j); // lane j holds the diagonal
      if (!(d > 0.0))
        fail = 1;
      const double rinv = rsqrt(d);
      if (i >= j && i < R)
        Hs[i + j * LD] = si * rinv; // the diagonal becomes d * rsqrt(d) = sqrt(d)
      if (i == j)
        inv[j] = rinv;
      __syncwarp();
    }
    return fail;
  }
#pragma unroll 1
  for (int j = 0; j < R; j++) {
    double rinv = 0.0;
#pragma unroll 1
    for (int i0 = j; i0 < R; i0 += 32) {
      const int i = i0 + lane;
      double a0 = 0.0, a1 = 0.0;
      if (i < R) {
        a0 = Hs[i + j * LD];
        const double *li = Hs + i, *lj = Hs + j;
        int k = 0;
#pragma unroll 2
        for (; k + 2 <= j; k += 2) {
          a0 -= li[k * LD] * lj[k * LD];
          a1 -= li[(k + 1) * LD] * lj[(k + 1) * LD];
        }
        if (k < j)
          a0 -= li[k * LD] * lj[k * LD];
      }
      const double si = a0 + a1;
      if (i0 == j) { // the pass that holds the diagonal (lane 0)
        const double d = __shfl_sync(0xffffffffu, si, 0);
        if (!(d > 0.0))
          fail = 1;
        rinv = rsqrt(d);
        if (lane == 0)
          inv[j] = rinv;
      }
      if (i < R)
        Hs[i + j * LD] = si * rinv;
    }
    __syncwarp();
  }
  return fail;
}

// Inverses of the 8 x 8 diagonal blocks of L, D_b = (L_bb)^-1 (lower triangular), written to the same positions of Di
// (ld = LD; everything else in Di stays zero).  Lane (blk, c) owns column c of block blk, four blocks per pass; the
// depth is 7 steps whatever the rank.
//   D[c][c] = inv[c],   D[i][c] = -inv[i] * sum_{k=c}^{i-1} L[i][k] D[k][c]
__device__ __forceinline__ void diag_block_inverses_warp(const double *L, int LD, const double *inv, double *Di, int R,
                                                         int lane) {
  const int NB = (R + 7) >> 3;
#pragma unroll 1
  for (int b0 = 0; b0 < NB; b0 += 4) {
    const int b = b0 + (lane >> 3), c = 8 * b + (lane & 7);
    if (b < NB && c < R) {
      double *x = Di + (size_t)c * LD;
      x[c] = inv[c];
      const int i_end = min(8 * b + 8, R);
#pragma unroll 1
      for (int i = c + 1; i < i_end; i++) {
        double acc = 0.0;
#pragma unroll 1
        for (int k = c; k < i; k++)
          acc += L[i + k * LD] * x[k];
        x[i] = -acc * inv[i];
      }
    }
  }
  __syncwarp();
}

// F = G H^-1 = (G L^-T) L^-1 for the rows staged in S (column-major, pitch = 4 mod 16 doubles so that the A fragments
// are bank-conflict free; columns R .. LD-1 zeroed), in place, as a blocked triangular solve on the FP64 tensor cores
// (mma.sync m8n8k4): with 8-column blocks,
//   forward   Y_b = (G_b - sum_{a<b} Y_a L_ba^T) D_b^T          b = 0 .. NB-1
//   backward  X_b = (Y_b - sum_{a>b} X_a L_ab  ) D_b            b = NB-1 .. 0
// Per-row substitution (thread per row) moves 16 bytes of shared memory per FMA and is bound by that pipe (measured
// 18.7 k cycles for 200 x 20); a DMMA moves 2.  Only the 8 x 8 diagonal blocks are inverted, so every product has the
// forward error of an 8 x 8 substitution.  Warp w owns the m8 row groups w, w + nw, ..; four of them are worked on at a
// time (independent accumulators, one B fragment for all four).  The loops carry no masks: the matrices are zero-padded
// to LD, rows of the last m8 group beyond nr compute garbage that nothing reads (rows of an MMA are independent).
constexpr int SOLVE_MB = 4;
__device__ __forceinline__ void solve_rows_dmma(double *S, int pitch, int nr, const double *L, const double *Di, int LD,
                                                int warp, int nw, int lane) {
  const int r = lane >> 2, s = lane & 3;
  const int MG = (nr + 7) >> 3, NB = LD >> 3;
#pragma unroll 1
  for (int mg0 = warp; mg0 < MG; mg0 += SOLVE_MB * nw) {
    double *Srow[SOLVE_MB];
    bool ok[SOLVE_MB];
#pragma unroll
    for (int g = 0; g < SOLVE_MB; g++) {
      ok[g] = (mg0 + g * nw) < MG;
      Srow[g] = S + 8 * (ok[g] ? mg0 + g * nw : mg0) + r; // a group beyond MG recomputes the first one, nothing stored
    }
#pragma unroll 1
    for (int dir = 0; dir < 2; dir++) { // 0: forward over L^T, 1: backward over L
#pragma unroll 1
      for (int bb = 0; bb < NB; bb++) {
        const int b = dir == 0 ? bb : NB - 1 - bb;
        double c0[SOLVE_MB], c1[SOLVE_MB];
#pragma unroll
        for (int g = 0; g < SOLVE_MB; g++)
          c0[g] = c1[g] = 0.0;
        // blocks already solved: a < b (forward), a > b (backward)
        const int k_lo = dir == 0 ? 0 : 8 * (b + 1), k_hi = dir == 0 ? 8 * b : LD;
        const int nb = 8 * b + r; // this lane's column of the B fragment
        // forward: B[k][n] = L[8b+n][k] -> L + nb + k * LD;  backward: B[k][n] = L[k][8b+n] -> L + k + nb * LD
        const double *bp = dir == 0 ? L + nb + (k_lo + s) * LD : L + (k_lo + s) + nb * LD;
        const int bstep = dir == 0 ? 4 * LD : 4;
#pragma unroll 1
        for (int k = k_lo + s; k < k_hi; k += 4, bp += bstep) {
          const double bf = *bp;
#pragma unroll
          for (int g = 0; g < SOLVE_MB; g++)
            dmma_m8n8k4(c0[g], c1[g], Srow[g][k * pitch], bf);
        }
        // T = (G_b or Y_b) - C, written back in place (accumulator layout: row r, columns 2s, 2s + 1)
        const int col = 8 * b + 2 * s;
#pragma unroll
        for (int g = 0; g < SOLVE_MB; g++)
          if (ok[g]) {
            Srow[g][col * pitch] -= c0[g];
            Srow[g][(col + 1) * pitch] -= c1[g];
          }
        __syncwarp();
        // times the inverse of the diagonal block: forward B[k][n] = D[n][k], backward B[k][n] = D[k][n] (the other
        // triangle of the block is zero)
#pragma unroll
        for (int g = 0; g < SOLVE_MB; g++)
          c0[g] = c1[g] = 0.0;
#pragma unroll
        for (int kk = 0; kk < 2; kk++) {
          const int k = 8 * b + 4 * kk + s;
          const double bf = dir == 0 ? Di[nb + k * LD] : Di[k + nb * LD];
#pragma unroll
          for (int g = 0; g < SOLVE_MB; g++)
            dmma_m8n8k4(c0[g], c1[g], Srow[g][k * pitch], bf);
        }
        __syncwarp(); // every lane has read T before it is overwritten
#pragma unroll
        for (int g = 0; g < SOLVE_MB; g++)
          if (ok[g]) {
            Srow[g][col * pitch] = c0[g];
            Srow[g][(col + 1) * pitch] = c1[g];
          }
        __syncwarp();
      }
    }
  }
}

// Gs += F^T F for the rows staged in S (pad columns zero), on the FP64 tensor cores: the 8 x 8 tiles of the lower block
// triangle (ti >= tj) are dealt to the warps; a tile's k loop runs over the rows with two accumulator pairs.  The scalar
// version (thread per entry) reads two shared-memory operands per FMA and is bound by that pipe (8.6 k cycles for
// 200 x 20).
__device__ __forceinline__ void gram_dmma(const double *S, int pitch, int nr, double *Gs, int LD, int warp, int nw,
                                          int lane) {
  const int r = lane >> 2, s = lane & 3, NT = LD >> 3;
  const int n_tiles = NT * (NT + 1) / 2;
#pragma unroll 1
  for (int t = warp; t < n_tiles; t += nw) {
    int ti = 0;
    while ((ti + 1) * (ti + 2) / 2 <= t)
      ti++;
    const int tj = t - ti * (ti + 1) / 2;
    const double *pa = S + (size_t)(8 * ti + r) * pitch + s, *pb = S + (size_t)(8 * tj + r) * pitch + s;
    double c0 = 0.0, c1 = 0.0, d0 = 0.0, d1 = 0.0;
    int k0 = 0;
#pragma unroll 2
    for (; k0 + 8 <= nr; k0 += 8) {
      dmma_m8n8k4(c0, c1, pa[k0], pb[k0]);
      dmma_m8n8k4(d0, d1, pa[k0 + 4], pb[k0 + 4]);
    }
#pragma unroll 1
    for (; k0 < nr; k0 += 4) {
      const bool okk = k0 + s < nr;
      dmma_m8n8k4(c0, c1, okk ? pa[k0] : 0.0, okk ? pb[k0] : 0.0);
    }
    double *gp = Gs + (8 * ti + r) + (8 * tj + 2 * s) * LD;
    gp[0] += c0 + d0;
    gp[LD] += c1 + d1;
  }
}

// The head of the update of mode n -- H = hadamard of the other modes' Gramians, its Cholesky factor, the inverses of the
// diagonal blocks -- depends on nothing the MTTKRP of mode n produces.  prefactor_kernel computes it for every live model
// on a forked branch of the iteration graph, next to the last light kernel in front of the update (the partial-tile
// reduction or the leaf that streams T), and model_update_kernel picks the result up from global memory: 17 k of its
// 34 k cycles (R = 20) leave the critical path.  Tuning knob (CALS_B200_PREFACTOR=1), off by default: on the B200 the
// extra graph edges and the contention with the leaf kernel cost more than that (engine.cu).  One CTA per live model; layout per slot: [H / L (LD x LD) | block
// inverses (LD x LD) | 1 / diag(L) (LD) | diag(H) (LD) | 1.0 if a pivot was not positive].
constexpr int PREFACTOR_THREADS = 128;
__global__ void __launch_bounds__(PREFACTOR_THREADS) prefactor_kernel(const PrefactorParams p) {
  const int n_live = p.st->n_live, m = p.live[blockIdx.x];
  if ((int)blockIdx.x >= n_live)
    return;
  const ModelDesc &md = p.models[m];
  if (md.rank > p.max_rank) // a wide model: wide.cuh
    return;
  const int R = md.rank, n = p.mode, N = p.n_modes;
  const int LD = (R + 7) & ~7;
  const int tid = threadIdx.x, nthr = blockDim.x;
  extern __shared__ double psm[];
  double *Hs = psm, *Gs = Hs + LD * LD, *inv = Gs + LD * LD, *hdiag = inv + LD;
  const double *grams = p.gram_pool + md.gram_off;
#pragma unroll 1
  for (int e = tid; e < LD * LD; e += nthr) {
    const int i = e % LD, j = e / LD;
    double h = 0.0;
    if (i < R && j < R) {
      h = 1.0;
#pragma unroll 1
      for (int k = 0; k < N; k++)
        if (k != n)
          h *= grams[(size_t)k * R * R + i + j * R];
      if (i == j)
        hdiag[i] = h;
    }
    Hs[e] = h;
    Gs[e] = 0.0;
  }
  for (int e = tid; e < LD; e += nthr) {
    inv[e] = 0.0;
    if (e >= R)
      hdiag[e] = 0.0;
  }
  __syncthreads();
  if (tid < 32) {
    const int fail = cholesky_warp(Hs, LD, inv, R, tid);
    diag_block_inverses_warp(Hs, LD, inv, Gs, R, tid);
    if (tid == 0) // non-positive pivot: the update kernel counts it in chol_info
      p.pref[(size_t)blockIdx.x * p.pref_stride + 2 * LD * LD + 2 * LD] = fail ? 1.0 : 0.0;
  }
  __syncthreads();
  double *out = p.pref + (size_t)blockIdx.x * p.pref_stride;
  for (int e = tid; e < 2 * LD * LD + 2 * LD; e += nthr)
    out[e] = psm[e];
}

constexpr int STAT_SEGS = 8; // row segments per column in the column statistics

template <bool NNLS>
__global__ void __launch_bounds__(UPDATE_THREADS, 2)
model_update_kernel(const UpdateParams p) {
  pdl_enter();
  SchedState *st = p.st;
  // both loads are issued before the branch (live[] has an entry for every CTA of the grid): one round trip to L2 less
  // on the dependent chain n_live -> live[b] -> model descriptor -> Gramians at the head of this latency-bound kernel
  const int n_live = st->n_live, m = p.live[blockIdx.x];
  if ((int)blockIdx.x >= n_live)
    return;
  ModelDesc &md = p.models[m];
  if (md.rank > p.max_rank) // a wide model: updated by the kernels of wide.cuh
    return;
  const int R = md.rank, col = md.col, cur = st->cur;
  const int rows = p.rows, ld = p.ld, n = p.mode, N = p.n_modes;
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int warp = tid >> 5, lane = tid & 31, nw = nthr >> 5;
  const int iters = md.iters;

  CALS_PROF(0);
  extern __shared__ double sm[];
  const int LD = (R + 7) & ~7;     // leading dimension of the small matrices (zero padding beyond R)
  double *Hs = sm;                 // LD x LD : H; the Cholesky factor takes its lower triangle, the strict upper keeps H
  double *Gs = Hs + LD * LD;       // LD x LD : inverses of L's diagonal blocks during pass 1, then the new Gramian
  double *cstat = Gs + LD * LD;    // 2R : per column reduction value / index ; then lambda, 1/lambda
  double *inv = cstat + 2 * R;     // R : 1 / L[j][j]
  double *hdiag = inv + R;         // R : diagonal of H (overwritten in Hs by the factorisation)
  double *red = hdiag + R;         // 64
  double *cand = red + 64;         // 2 * STAT_SEGS * R : per (column, row segment) candidates of the column statistics
  double *S = cand + 2 * STAT_SEGS * R; // chunk_rows x R, pitch chunk_pitch
  const int pitch = p.chunk_pitch, CR = p.chunk_rows;
  // NNLS scratch (only allocated when p.nnls): per working warp 5R + R*R doubles and 2R + 1 ints, behind S
  double *nn_base = S + (size_t)pitch * ((p.max_rank + 7) & ~7);
  // tile lookup tables of the fused partial-tile reduction: R + chunk_rows ints at the very end of the allocation
  int *cinfo = reinterpret_cast<int *>(sm + p.table_off);
  int *rinfo = cinfo + p.max_rank;

  double *grams = p.gram_pool + md.gram_off;
  const double *Gm = p.G + (size_t)col * ld;
  double *Fm = p.F[cur] + (size_t)col * ld;
  const bool fused = p.plan != nullptr;
  const PlanView pv = fused ? plan_view(p.plan, p.plan_ctas) : PlanView{};

  // ---- H = hadamard of the other Gramians (or everything prefactor_kernel has derived from it) ----
  const bool prefactored = !NNLS && p.pref != nullptr;
  int chol_fail = 0;
  if (prefactored) {
    const double *src = p.pref + (size_t)blockIdx.x * p.pref_stride;
    for (int e = tid; e < 2 * LD * LD; e += nthr)
      Hs[e] = src[e]; // Hs and Gs are adjacent
    for (int e = tid; e < R; e += nthr) {
      inv[e] = src[2 * LD * LD + e];
      hdiag[e] = src[2 * LD * LD + LD + e];
    }
    chol_fail = src[2 * LD * LD + 2 * LD] != 0.0;
  } else {
#pragma unroll 1
    for (int e = tid; e < LD * LD; e += nthr) {
      const int i = e % LD, j = e / LD;
      double h = 0.0;
      if (i < R && j < R) {
        h = 1.0;
#pragma unroll 1
        for (int k = 0; k < N; k++)
          if (k != n)
            h *= grams[(size_t)k * R * R + i + j * R];
        if (i == j)
          hdiag[i] = h;
      }
      Hs[e] = h;
      Gs[e] = 0.0;
    }
  }
  for (int e = tid; e < 2 * R; e += nthr) // value: a sum of squares starts at 0, a max-abs at -1; then the index
    cstat[e] = (e < R) ? (iters == 1 ? 0.0 : -1.0) : 0.0;
  if (fused) // (n-tile, column in tile) of every column of the model
    for (int j = tid; j < R; j += nthr) {
      const int cg = col + j;
      const int nt = plan_tile_of(cg >> 6, pv.NO, pv.n_tiles);
      cinfo[j] = (nt << 8) | (cg - 64 * plan_oct_start(nt, pv.NO, pv.n_tiles));
    }
  __syncthreads();
  CALS_PROF(1);

  double nnls_tol = 0.0;
  if (NNLS) { // tol = 10 * eps * ||H||_1 * R   (reference src/utils/update.cpp:65-66; one_norm = max column sum)
    double mx = -1.0;
    for (int j = tid; j < R; j += nthr) {
      double cs = 0.0;
      for (int i = 0; i < R; i++)
        cs += fabs(Hs[i + j * LD]);
      mx = fmax(mx, cs);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
      mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0)
      red[warp] = mx;
    __syncthreads();
    mx = red[0];
    for (int wv = 1; wv < nw; wv++)
      mx = fmax(mx, red[wv]);
    nnls_tol = 10 * 2.2204e-16 * mx * (double)R;
    __syncthreads();
  }

  const bool jk_here = (md.jk_mode == n);
  const int jk_row = md.jk_fiber;
  const bool single = rows <= CR;

  // ---- pass 1: Cholesky || staging, solve rows, jackknife row, column statistics ----
#pragma unroll 1
  for (int r0 = 0; r0 < rows; r0 += CR) {
    const int nr = min(CR, rows - r0);
    if (r0 > 0)
      __syncthreads(); // S and rinfo are free again
    if (fused) {       // (m-tile, row in tile) of every row of the chunk
      for (int rr = tid; rr < nr; rr += nthr) {
        const int mrow = r0 + rr;
        const int mt = plan_tile_of(mrow >> 3, pv.In8, pv.m_tiles);
        rinfo[rr] = (mt << 8) | (mrow - 8 * plan_m8_start(mt, pv.In8, pv.m_tiles));
      }
      __syncthreads();
    }
    // Stage rows [r0, r0 + nr) of the MTTKRP result into S.  In the first chunk warp 0 factors H meanwhile (and inverts
    // the diagonal blocks of L); the other warps stage.
    const bool overlap = r0 == 0 && !NNLS && !prefactored;
    if (overlap && warp == 0) {
      chol_fail = cholesky_warp(Hs, LD, inv, R, lane);
      diag_block_inverses_warp(Hs, LD, inv, Gs, R, lane);
      CALS_PROF(2);
    } else if (fused) {
      // Fused reduction: the result is not read from G but summed here, per (m,n) pair in segment order with four
      // running sums, from the partial tiles the DMMA kernel has just written; for the last mode the sum also goes to
      // G (the error term needs it after the solve).  Columns fastest: runs of R doubles of a row-major tile.
      const int t0 = overlap ? tid - 32 : tid, tn = overlap ? nthr - 32 : nthr;
      double *Gw = p.G_out + (size_t)col * ld;
      const int dj = tn % R, dr = tn / R;
      int j = t0 % R, rr = t0 / R;
#pragma unroll 1
      while (rr < nr) {
        const int ci = cinfo[j], ri = rinfo[rr];
        const int pair = (ci >> 8) * pv.m_tiles + (ri >> 8);
        const int s0 = pv.pair_seg0[pair], s1 = pv.pair_seg0[pair + 1];
        const double *q = p.ws + (size_t)s0 * p.tile_elems + (size_t)(ri & 255) * p.n_tile + (ci & 255);
        const size_t te = (size_t)p.tile_elems;
        double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
        int k = s0;
#pragma unroll 1
        for (; k + 4 <= s1; k += 4, q += 4 * te) {
          a0 += q[0];
          a1 += q[te];
          a2 += q[2 * te];
          a3 += q[3 * te];
        }
#pragma unroll 1
        for (; k < s1; k++, q += te)
          a0 += *q;
        const double sum = (a0 + a1) + (a2 + a3);
        S[rr + j * pitch] = sum;
        if (n == N - 1) // keep G for the error term
          Gw[(size_t)j * ld + r0 + rr] = sum;
        j += dj;
        rr += dr;
        if (j >= R) {
          j -= R;
          rr++;
        }
      }
    } else {
      const int w0 = overlap ? warp - 1 : warp, wn = overlap ? nw - 1 : nw;
#pragma unroll 1
      for (int j = w0; j < R; j += wn) {
        const double *gj = Gm + (size_t)j * ld + r0;
        double *sj = S + j * pitch;
#pragma unroll 2
        for (int rr = lane; rr < nr; rr += 32)
          sj[rr] = gj[rr];
      }
    }
    if (!(overlap && warp == 0)) { // columns R .. LD-1 of the staged chunk: zero (the tensor-core loops read them)
      const int t0 = overlap ? tid - 32 : tid, tn = overlap ? nthr - 32 : nthr;
      for (int e = t0; e < (LD - R) * nr; e += tn)
        S[(e % nr) + (R + e / nr) * pitch] = 0.0;
    }
    __syncthreads();
    CALS_PROF(3);
    if (NNLS) { // warp per row, active sets warm-started from the previous iteration
      if (warp < p.nnls_warps) {
        const size_t per_warp = (size_t)5 * R + (size_t)R * R + (size_t)(2 * R + 2) / 2 + 1; // doubles
        double *wb = nn_base + per_warp * warp;
        NnlsScratch q;
        q.y = wb;
        q.d = wb + R;
        q.w = wb + 2 * R;
        q.s = wb + 3 * R;
        q.sp = wb + 4 * R;
        q.Gp = wb + 5 * R;
        q.act = reinterpret_cast<int *>(wb + 5 * R + (size_t)R * R);
        q.map = q.act + R;
        unsigned char *act = p.act_pool + md.act_off + (size_t)p.rows_before * R;
        int trouble = 0;
        for (int rr = warp; rr < nr; rr += p.nnls_warps)
          trouble += nnls_row(Hs, LD, R, nnls_tol, S + rr, pitch, act + (size_t)(r0 + rr) * R, q, lane);
        if (trouble && lane == 0)
          chol_fail = 1;
      }
    } else {
      solve_rows_dmma(S, pitch, nr, Hs, Gs, LD, warp, nw, lane);
    }
    __syncthreads();
    CALS_PROF(4);
    if (jk_here && jk_row >= r0 && jk_row < r0 + nr) { // Ktensor::set_jk_fiber(0.0)
      for (int j = tid; j < R; j += nthr)
        S[(jk_row - r0) + j * pitch] *= 0.0;
      __syncthreads();
    }
    // Column statistics (Ktensor::normalize, src/ktensor.cpp:66-83): sum of squares at the model's first iteration, else
    // the entry of largest magnitude with the first index on ties.  Thread (column, segment) scans one of STAT_SEGS
    // row segments; the segments of a column are then combined in row order.
    {
      const int seg = tid % STAT_SEGS, seg_len = (nr + STAT_SEGS - 1) / STAT_SEGS;
      const int lo = seg * seg_len, hi = min(nr, lo + seg_len);
#pragma unroll 1
      for (int j = tid / STAT_SEGS; j < R; j += nthr / STAT_SEGS) {
        const double *cj = S + j * pitch;
        double v = iters == 1 ? 0.0 : -1.0;
        int bi = 0x7fffffff;
        if (iters == 1) {
#pragma unroll 2
          for (int rr = lo; rr < hi; rr++)
            v += cj[rr] * cj[rr];
        } else {
#pragma unroll 2
          for (int rr = lo; rr < hi; rr++) {
            const double a = fabs(cj[rr]);
            if (a > v) { // strictly greater keeps the first index
              v = a;
              bi = r0 + rr;
            }
          }
        }
        cand[(j * STAT_SEGS + seg) * 2] = v;
        cand[(j * STAT_SEGS + seg) * 2 + 1] = (double)bi;
      }
      __syncthreads();
      for (int j = tid; j < R; j += nthr) {
        const double *cj = cand + (size_t)j * STAT_SEGS * 2;
        if (iters == 1) {
          double ss = 0.0;
          for (int q = 0; q < STAT_SEGS; q++)
            ss += cj[2 * q];
          cstat[j] += ss;
        } else {
          double best = cstat[j], bidx = cstat[R + j]; // earlier chunks / segments win ties (first index, as idamax)
          for (int q = 0; q < STAT_SEGS; q++)
            if (cj[2 * q] > best) {
              best = cj[2 * q];
              bidx = cj[2 * q + 1];
            }
          cstat[j] = best;
          cstat[R + j] = bidx;
        }
      }
    }
    if (!single) {
      __syncthreads();
#pragma unroll 1
      for (int j = warp; j < R; j += nw)
        for (int rr = lane; rr < nr; rr += 32)
          Fm[(size_t)j * ld + r0 + rr] = S[rr + j * pitch];
    }
  }
  __syncthreads();
  CALS_PROF(5);

  // ---- lambda ----
  for (int e = tid; e < LD * LD; e += nthr) // the block inverses are done with; from here on the new Gramian accumulates
    Gs[e] = 0.0;
  for (int j = tid; j < R; j += nthr) {
    double lam;
    if (iters == 1)
      lam = sqrt(cstat[j]);
    else {
      const int bi = (int)cstat[R + j];
      lam = single ? S[bi + j * pitch] : Fm[(size_t)j * ld + bi];
    }
    p.lambda_home[md.home_col + j] = lam;
    cstat[j] = lam;
    cstat[R + j] = (lam != 0.0) ? 1.0 / lam : 1.0;
  }
  __syncthreads();
  CALS_PROF(6);

  // ---- pass 2: scale, write factor, accumulate Gramian (and <F, G> per column for the error) ----
  const bool last_mode = (n == N - 1);
  double term3 = 0.0;
#pragma unroll 1
  for (int r0 = 0; r0 < rows; r0 += CR) {
    const int nr = min(CR, rows - r0);
    if (r0 > 0)
      __syncthreads();
#pragma unroll 1
    for (int j = warp; j < R; j += nw) {
      double *sj = S + j * pitch;
      double *fj = Fm + (size_t)j * ld + r0;
      const double *gj = Gm + (size_t)j * ld + r0;
      const double lam = cstat[j], rl = cstat[R + j];
#pragma unroll 2
      for (int rr = lane; rr < nr; rr += 32) {
        const double v = (single ? sj[rr] : fj[rr]) * rl;
        sj[rr] = v;
        fj[rr] = v;
        if (last_mode)
          term3 += lam * v * gj[rr];
      }
    }
    __syncthreads();
    CALS_PROF(7);
    gram_dmma(S, pitch, nr, Gs, LD, warp, nw, lane);
  }
  __syncthreads();
  CALS_PROF(8);
  for (int e = tid; e < R * R; e += nthr) { // mirror, then publish
    const int i = e % R, j = e / R;
    const double v = (i >> 3) >= (j >> 3) ? Gs[i + j * LD] : Gs[j + i * LD]; // tiles of the lower block triangle
    grams[(size_t)n * R * R + e] = v;
  }
  if (__syncthreads_or(chol_fail) && tid == 0)
    md.chol_info += 1;
  CALS_PROF(9);
  if (p.prof != nullptr && tid == 0)
    p.prof[(size_t)blockIdx.x * 16 + 15] = R;

  if (!last_mode)
    return;

  // ---- fast error, fit, eviction decision ----
  // P = hadamard of all Gramians = H (the other modes; still in the strict upper triangle of Hs and in hdiag) times the
  // new Gramian of this mode
  double term2 = 0.0;
  for (int e = tid; e < R * R; e += nthr) {
    const int i = e % R, j = e / R;
    const double gn = (i >> 3) >= (j >> 3) ? Gs[i + j * LD] : Gs[j + i * LD];
    const double h = i == j ? hdiag[i] : (i < j ? Hs[i + j * LD] : Hs[j + i * LD]);
    term2 += cstat[i] * cstat[j] * h * gn;
  }
  // both sums with one pass through shared memory
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    term2 += __shfl_xor_sync(0xffffffffu, term2, o);
    term3 += __shfl_xor_sync(0xffffffffu, term3, o);
  }
  if (lane == 0) {
    red[warp] = term2;
    red[32 + warp] = term3;
  }
  __syncthreads();
  if (tid == 0) {
    term2 = term3 = 0.0;
    for (int wv = 0; wv < nw; wv++) {
      term2 += red[wv];
      term3 += red[32 + wv];
    }
    double xn = st->x_norm;
    if (md.jk_mode >= 0 && p.x_norms_jk)
      xn = p.x_norms_jk[md.jk_fiber];
    const double err = sqrt(fmax(xn * xn + term2 - 2.0 * term3, 0.0));
    const double old_fit = md.fit;
    const double fit = 1.0 - fabs(err) / st->x_norm;
    md.error = err;
    md.old_fit = old_fit;
    md.fit = fit;
    if (!st->ls_enabled) // with line search the decision is taken after the extrapolation step (ls.cuh)
      decide_eviction(md, st);
    CALS_PROF(10);
  }
}

// Gramians of the incoming factors of every queued model (MultiKtensor::add computes them on admission,
// reference src/multi_ktensor.cpp:89-95; here all at once before the loop starts).  One CTA per (model, mode).
__global__ void __launch_bounds__(256)
init_grams_kernel(const Geom geo, const FactorPtrs fac, const ModelDesc *__restrict__ models, double *gram_pool) {
  const int m = blockIdx.x, n = blockIdx.y;
  const ModelDesc &md = models[m];
  const int R = md.rank, rows = geo.dims[n], ld = geo.ldF[n];
  const double *F = fac.home[n] + (size_t)md.home_col * ld;
  double *gr = gram_pool + md.gram_off + (size_t)n * R * R;
  for (int e = threadIdx.x; e < R * R; e += blockDim.x) {
    const int i = e % R, j = e / R;
    const double *ci = F + (size_t)i * ld, *cj = F + (size_t)j * ld;
    double g = 0.0;
    for (int r = 0; r < rows; r++)
      g += ci[r] * cj[r];
    gr[e] = g;
  }
}

} // namespace calsb200
