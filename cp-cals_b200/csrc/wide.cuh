// Update of models whose rank is above what the one-CTA shared-memory kernel (update.cuh: model_update_kernel) can hold.
// Same work and the same reference lines as that kernel (see update.cuh:1-13), split over several kernels per mode that
// keep the R x R matrices in a global workspace (one slot per concurrently live wide model, L2-resident for R <= 1024):
//
//   wide_factor_kernel   one thread-block cluster per model: H = hadamard of the other Gramians, blocked right-looking
//                        Cholesky H = L L^T (64-column panels; the diagonal block is factored redundantly by every CTA
//                        of the cluster, panel and trailing DMMA updates are dealt to the CTAs), then L^-1 by blocked
//                        forward substitution, one 64-column block of L^-1 per CTA (the column blocks are independent)
//   wide_solve_kernel    Y = G L^-T, then (second launch) F = Y L^-1: 64 x 64 DMMA tiles over rows and columns
//   wide_stats_kernel    jackknife row, column statistics, lambda, scaling (a warp owns whole columns); <F, G> per column
//                        on the last mode
//   wide_gram_kernel     Gram_n = F^T F, one 64 x 64 tile of the lower block triangle per CTA, mirrored
//   wide_error_kernel    last mode: fast error, fit, eviction decision
//
// Every reduction runs in a fixed order without floating-point atomics, so a rerun is bit-identical.  The kernels find
// their model from the device-side live set: the s-th live model of rank above `bound` (in live order) uses slot s.
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include "common.cuh"
#include "mttkrp.cuh"
#include "update.cuh"

namespace calsb200 {

constexpr int WIDE_NB = 64;      // block size of the factorisation and tile size of every DMMA loop
constexpr int WIDE_TP = 68;      // pitch (doubles) of a 64 x 64 tile in shared memory, = 4 mod 16
constexpr int WIDE_CLUSTER = 8;  // CTAs per model in wide_factor_kernel (portable cluster size)
constexpr int WIDE_THREADS = 256; // every wide kernel: 8 warps, warp w owns rows 8w .. 8w + 7 of a 64 x 64 tile
constexpr int WIDE_TILE = WIDE_NB * WIDE_TP;
constexpr size_t WIDE_FACTOR_SMEM = (size_t)(4 * WIDE_TILE + WIDE_NB) * 8;
constexpr size_t WIDE_TILE_SMEM = (size_t)2 * WIDE_TILE * 8;

struct WideParams {
  int mode, n_modes;
  int rows, ld;        // I_n, ldF[n] (== ld of G)
  int bound;           // a model is wide when its rank is above this
  const double *G;     // MTTKRP result, ld x C
  double *F[2];        // multi-factor buffers of this mode
  double *gram_pool;
  double *lambda_home;
  const double *x_norms_jk;
  ModelDesc *models;
  const int *live;
  SchedState *st;
  // workspace, per slot: H | L | L^-1 (ldw x ldw each) | Y (y_rows x ldw) | lambda (ldw) | <F, G> per column (ldw)
  double *ws;
  long long slot_stride;
  int ldw;    // wide ranks rounded up to 64, largest of the run
  int y_rows; // I_n rounded up to 64, largest of the run
};

struct WideSlot {
  double *H, *L, *Li, *Y, *lam, *t3;
};

__device__ __forceinline__ WideSlot wide_slot(const WideParams &p, int slot) {
  WideSlot w;
  const size_t m2 = (size_t)p.ldw * p.ldw;
  w.H = p.ws + (size_t)slot * p.slot_stride;
  w.L = w.H + m2;
  w.Li = w.L + m2;
  w.Y = w.Li + m2;
  w.lam = w.Y + (size_t)p.y_rows * p.ldw;
  w.t3 = w.lam + p.ldw;
  return w;
}

// the current factor buffer of this mode (a select: indexing the parameter array with a run-time value would copy it to
// local memory)
__device__ __forceinline__ double *wide_factor(const WideParams &p) { return p.st->cur ? p.F[1] : p.F[0]; }

// The model of slot `slot`: the slot-th live model of rank > bound, in live order, or -1.  Block-wide scan, the same
// result in every CTA; all threads must call it.
__device__ int wide_find_model(const WideParams &p, int slot) {
  __shared__ int s_cnt[WIDE_THREADS / 32];
  __shared__ int s_res;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_live = p.st->n_live;
  if (tid == 0)
    s_res = -1;
  int seen = 0;
  for (int base = 0; base < n_live; base += WIDE_THREADS) {
    const int i = base + tid;
    const int m = i < n_live ? p.live[i] : -1;
    const bool wide = m >= 0 && p.models[m].rank > p.bound;
    const unsigned bal = __ballot_sync(0xffffffffu, wide);
    if (lane == 0)
      s_cnt[warp] = __popc(bal);
    __syncthreads();
    int before = seen, total = 0;
    for (int w = 0; w < WIDE_THREADS / 32; w++) {
      before += w < warp ? s_cnt[w] : 0;
      total += s_cnt[w];
    }
    if (wide && before + __popc(bal & ((1u << lane) - 1u)) == slot)
      s_res = m;
    seen += total;
    __syncthreads();
    if (seen > slot)
      break;
  }
  __syncthreads();
  return s_res;
}

// 64 x 64 tile product on the FP64 tensor cores (mma.sync m8n8k4): acc += op(A) op(B) over k = 0 .. 63, with
//   op(A)(i, k) = TA ? A[k + i * TP] : A[i + k * TP],   op(B)(k, j) = TB ? B[j + k * TP] : B[k + j * TP].
// Warp w owns rows 8w .. 8w + 7 and all eight n8 groups: acc[j][0..1] = C[8w + r][8j + 2s, 8j + 2s + 1].
template <bool TA, bool TB>
__device__ __forceinline__ void wide_tile_mma(double (&acc)[8][2], const double *A, const double *B, int warp, int lane) {
  const int r = lane >> 2, s = lane & 3, i = 8 * warp + r;
#pragma unroll 4
  for (int k0 = 0; k0 < WIDE_NB; k0 += 4) {
    const int k = k0 + s;
    const double a = TA ? A[k + i * WIDE_TP] : A[i + k * WIDE_TP];
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const int n = 8 * j + r;
      const double b = TB ? B[n + k * WIDE_TP] : B[k + n * WIDE_TP];
      dmma_m8n8k4(acc[j][0], acc[j][1], a, b);
    }
  }
}

__device__ __forceinline__ void wide_acc_zero(double (&acc)[8][2]) {
#pragma unroll
  for (int j = 0; j < 8; j++)
    acc[j][0] = acc[j][1] = 0.0;
}

// tile <- global block at (r0, c0) of a column-major matrix with leading dimension ld; entries with row >= nr or
// column >= nc read as zero.  Loads bypass L1 (other CTAs of the cluster write the workspace).
__device__ __forceinline__ void wide_stage(double *t, const double *src, size_t ld, int r0, int c0, int nr, int nc) {
  for (int e = threadIdx.x; e < WIDE_NB * WIDE_NB; e += WIDE_THREADS) {
    const int i = e & (WIDE_NB - 1), j = e >> 6;
    const int gi = r0 + i, gj = c0 + j;
    t[i + j * WIDE_TP] = (gi < nr && gj < nc) ? __ldcg(src + gi + (size_t)gj * ld) : 0.0;
  }
}

// the warp's accumulator -> tile in shared memory (scaled by `sign`)
__device__ __forceinline__ void wide_acc_to_tile(double *t, const double (&acc)[8][2], double sign, int warp, int lane) {
  const int r = lane >> 2, s = lane & 3, i = 8 * warp + r;
#pragma unroll
  for (int j = 0; j < 8; j++) {
    t[i + (8 * j + 2 * s) * WIDE_TP] = sign * acc[j][0];
    t[i + (8 * j + 2 * s + 1) * WIDE_TP] = sign * acc[j][1];
  }
}

// the warp's accumulator -> global block at (r0, c0), rows < nr and columns < nc only
__device__ __forceinline__ void wide_acc_store(double *dst, size_t ld, int r0, int c0, int nr, int nc,
                                               const double (&acc)[8][2], int warp, int lane) {
  const int r = lane >> 2, s = lane & 3, gi = r0 + 8 * warp + r;
  if (gi >= nr)
    return;
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const int gj = c0 + 8 * j + 2 * s;
    if (gj < nc)
      dst[gi + (size_t)gj * ld] = acc[j][0];
    if (gj + 1 < nc)
      dst[gi + (size_t)(gj + 1) * ld] = acc[j][1];
  }
}

// Factor the 64 x 64 diagonal block in sA (pitch WIDE_TP) in place (lower triangle = L_kk) and write its inverse to sD
// (lower triangular, upper triangle zero).  Warp 0 factors (cholesky_warp) and inverts the 8 x 8 diagonal blocks; then
// warp w forms the column block w of the inverse by blocked forward substitution,
//   X_bw = -D_b sum_{w <= a < b} L_ba X_aw,   b = w + 1 .. 7  (D_b = inverse of the 8 x 8 diagonal block b).
// Returns 1 (in every thread) when a pivot was not positive.
__device__ int wide_factor_diag(double *sA, double *sD, double *inv, int *fail_flag) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int e = tid; e < WIDE_TILE; e += WIDE_THREADS)
    sD[e] = 0.0;
  __syncthreads();
  if (warp == 0) {
    const int f = cholesky_warp(sA, WIDE_TP, inv, WIDE_NB, lane);
    diag_block_inverses_warp(sA, WIDE_TP, inv, sD, WIDE_NB, lane);
    if (lane == 0)
      *fail_flag = f;
  }
  __syncthreads();
  const int r = lane >> 2, s = lane & 3, w = warp;
#pragma unroll 1
  for (int b = w + 1; b < 8; b++) {
    double c0 = 0.0, c1 = 0.0;
    // sum_{k = 8w}^{8b - 1} L[8b + r][k] X[k][8w + n]
#pragma unroll 1
    for (int k0 = 8 * w; k0 < 8 * b; k0 += 4) {
      const int k = k0 + s;
      dmma_m8n8k4(c0, c1, sA[(8 * b + r) + k * WIDE_TP], sD[k + (8 * w + r) * WIDE_TP]);
    }
    // T = -C, kept in registers and exchanged through shuffles: lane (r, s) holds T[r][2s], T[r][2s + 1]; the second
    // product needs B[k][n] = T[k][n] at lane (n, k % 4) for k = s and k = s + 4
    double bt[2];
#pragma unroll
    for (int kk = 0; kk < 2; kk++) {
      const int k = 4 * kk + s, n = r;
      // owner of T[k][n]: lane (k, n / 2), register n % 2
      const int src = 4 * k + (n >> 1);
      const double v0 = __shfl_sync(0xffffffffu, c0, src), v1 = __shfl_sync(0xffffffffu, c1, src);
      bt[kk] = -((n & 1) ? v1 : v0);
    }
    double x0 = 0.0, x1 = 0.0;
#pragma unroll
    for (int kk = 0; kk < 2; kk++) {
      const int k = 4 * kk + s;
      dmma_m8n8k4(x0, x1, sD[(8 * b + r) + (8 * b + k) * WIDE_TP], bt[kk]);
    }
    sD[(8 * b + r) + (8 * w + 2 * s) * WIDE_TP] = x0;
    sD[(8 * b + r) + (8 * w + 2 * s + 1) * WIDE_TP] = x1;
    __syncwarp();
  }
  __syncthreads();
  return *fail_flag;
}

__device__ __forceinline__ void wide_cluster_sync() {
  __threadfence();
  cooperative_groups::this_cluster().sync();
}

// H, L and L^-1 of one wide model per cluster.  grid = (WIDE_CLUSTER, slots).
__global__ void __cluster_dims__(WIDE_CLUSTER, 1, 1) __launch_bounds__(WIDE_THREADS)
wide_factor_kernel(const WideParams p) {
  const int m = wide_find_model(p, blockIdx.y);
  if (m < 0)
    return; // the same in every CTA of the cluster
  ModelDesc &md = p.models[m];
  const int R = md.rank, n = p.mode, N = p.n_modes, ldw = p.ldw;
  const int NT = (R + WIDE_NB - 1) / WIDE_NB, RP = NT * WIDE_NB;
  const int cta = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const WideSlot w = wide_slot(p, blockIdx.y);
  extern __shared__ double wsm[];
  double *sA = wsm, *sD = sA + WIDE_TILE, *sB = sD + WIDE_TILE, *sC = sB + WIDE_TILE, *inv = sC + WIDE_TILE;
  __shared__ int fail_flag;

  // H (kept for the error term) and its copy that the factorisation overwrites; padded with the identity, so that L and
  // L^-1 are block diagonal with an identity block beyond R; L^-1 starts at zero
  const double *grams = p.gram_pool + md.gram_off;
  for (long long e = (long long)cta * WIDE_THREADS + tid; e < (long long)RP * RP; e += WIDE_CLUSTER * WIDE_THREADS) {
    const int i = (int)(e % RP), j = (int)(e / RP);
    double h;
    if (i < R && j < R) {
      h = 1.0;
      for (int k = 0; k < N; k++)
        if (k != n)
          h *= grams[(size_t)k * R * R + i + (size_t)j * R];
    } else
      h = i == j ? 1.0 : 0.0;
    const size_t o = i + (size_t)j * ldw;
    w.H[o] = h;
    w.L[o] = h;
    w.Li[o] = 0.0;
  }
  wide_cluster_sync();

  int fail = 0;
#pragma unroll 1
  for (int k = 0; k < NT; k++) {
    const int k0 = k * WIDE_NB;
    wide_stage(sA, w.L, ldw, k0, k0, RP, RP);
    __syncthreads();
    fail |= wide_factor_diag(sA, sD, inv, &fail_flag);
    if (cta == 0) // L^-1 of the diagonal block: the diagonal block of L^-1
      for (int e = tid; e < WIDE_NB * WIDE_NB; e += WIDE_THREADS) {
        const int i = e & (WIDE_NB - 1), j = e >> 6;
        w.Li[(k0 + i) + (size_t)(k0 + j) * ldw] = sD[i + j * WIDE_TP];
      }
    // panel: L_ik = A_ik L_kk^-T
#pragma unroll 1
    for (int i = k + 1 + cta; i < NT; i += WIDE_CLUSTER) {
      __syncthreads();
      wide_stage(sB, w.L, ldw, i * WIDE_NB, k0, RP, RP);
      __syncthreads();
      double acc[8][2];
      wide_acc_zero(acc);
      wide_tile_mma<false, true>(acc, sB, sD, warp, lane);
      wide_acc_store(w.L, ldw, i * WIDE_NB, k0, RP, RP, acc, warp, lane);
    }
    wide_cluster_sync();
    // trailing update of the lower block triangle: A_ij -= L_ik L_jk^T, k < j <= i
    const int T = NT - k - 1;
#pragma unroll 1
    for (int t = cta; t < T * (T + 1) / 2; t += WIDE_CLUSTER) {
      int ti = 0;
      while ((ti + 1) * (ti + 2) / 2 <= t)
        ti++;
      const int tj = t - ti * (ti + 1) / 2;
      const int i0 = (k + 1 + ti) * WIDE_NB, j0 = (k + 1 + tj) * WIDE_NB;
      __syncthreads();
      wide_stage(sB, w.L, ldw, i0, k0, RP, RP);
      wide_stage(sC, w.L, ldw, j0, k0, RP, RP);
      __syncthreads();
      double acc[8][2];
      wide_acc_zero(acc);
      wide_tile_mma<false, true>(acc, sB, sC, warp, lane);
      const int r = lane >> 2, s = lane & 3, gi = i0 + 8 * warp + r;
#pragma unroll
      for (int j = 0; j < 8; j++) {
        double *d = w.L + gi + (size_t)(j0 + 8 * j + 2 * s) * ldw;
        d[0] = __ldcg(d) - acc[j][0];
        d[ldw] = __ldcg(d + ldw) - acc[j][1];
      }
    }
    wide_cluster_sync();
  }
  if (cta == 0 && tid == 0 && fail) // dpotrf's info > 0: counted, the update carries on (as the narrow kernel)
    md.chol_info += 1;

  // L^-1, column block cb: X_cb = D_cb (done above), X_b = -D_b sum_{cb <= a < b} L_ba X_a
#pragma unroll 1
  for (int cb = cta; cb < NT; cb += WIDE_CLUSTER) {
    const int c0 = cb * WIDE_NB;
#pragma unroll 1
    for (int b = cb + 1; b < NT; b++) {
      double acc[8][2];
      wide_acc_zero(acc);
#pragma unroll 1
      for (int a = cb; a < b; a++) {
        __syncthreads();
        wide_stage(sB, w.L, ldw, b * WIDE_NB, a * WIDE_NB, RP, RP);
        wide_stage(sC, w.Li, ldw, a * WIDE_NB, c0, RP, RP);
        __syncthreads();
        wide_tile_mma<false, false>(acc, sB, sC, warp, lane);
      }
      __syncthreads();
      wide_acc_to_tile(sC, acc, -1.0, warp, lane);
      wide_stage(sA, w.Li, ldw, b * WIDE_NB, b * WIDE_NB, RP, RP);
      __syncthreads();
      wide_acc_zero(acc);
      wide_tile_mma<false, false>(acc, sA, sC, warp, lane);
      wide_acc_store(w.Li, ldw, b * WIDE_NB, c0, RP, RP, acc, warp, lane);
    }
  }
}

// pass 0: Y = G L^-T (G's columns beyond R and rows beyond I_n read as zero); pass 1: F = Y L^-1, written to the
// factor buffer.  grid = (row tiles x column tiles of the largest wide model, slots).
template <int PASS>
__global__ void __launch_bounds__(WIDE_THREADS) wide_solve_kernel(const WideParams p) {
  const int m = wide_find_model(p, blockIdx.y);
  if (m < 0)
    return;
  const ModelDesc &md = p.models[m];
  const int R = md.rank, NT = (R + WIDE_NB - 1) / WIDE_NB, RT = (p.rows + WIDE_NB - 1) / WIDE_NB;
  const int rt = blockIdx.x % RT, ct = blockIdx.x / RT;
  if (ct >= NT)
    return;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const WideSlot w = wide_slot(p, blockIdx.y);
  extern __shared__ double wsm[];
  double *sA = wsm, *sB = sA + WIDE_TILE;
  const int r0 = rt * WIDE_NB, c0 = ct * WIDE_NB;
  double acc[8][2];
  wide_acc_zero(acc);
  // pass 0: Y[r][j] = sum_{k <= j} G[r][k] L^-1[j][k];  pass 1: F[r][j] = sum_{k >= j} Y[r][k] L^-1[k][j]
  const int kt_lo = PASS == 0 ? 0 : ct, kt_hi = PASS == 0 ? ct + 1 : NT;
#pragma unroll 1
  for (int kt = kt_lo; kt < kt_hi; kt++) {
    __syncthreads();
    if (PASS == 0) {
      wide_stage(sA, p.G + (size_t)md.col * p.ld, p.ld, r0, kt * WIDE_NB, p.rows, R);
      wide_stage(sB, w.Li, p.ldw, c0, kt * WIDE_NB, R, R); // sB(j, k) = L^-1[c0 + j][k]
    } else {
      wide_stage(sA, w.Y, p.y_rows, r0, kt * WIDE_NB, p.rows, R);
      wide_stage(sB, w.Li, p.ldw, kt * WIDE_NB, c0, R, R); // sB(k, j) = L^-1[k][c0 + j]
    }
    __syncthreads();
    if (PASS == 0)
      wide_tile_mma<false, true>(acc, sA, sB, warp, lane);
    else
      wide_tile_mma<false, false>(acc, sA, sB, warp, lane);
  }
  if (PASS == 0)
    wide_acc_store(w.Y, p.y_rows, r0, c0, p.rows, R, acc, warp, lane);
  else
    wide_acc_store(wide_factor(p) + (size_t)md.col * p.ld, p.ld, r0, c0, p.rows, R, acc, warp, lane);
}

// Ktensor::set_jk_fiber(0) and Ktensor::normalize(n, it) for 32 columns per CTA (a warp per column, whole columns):
// sum of squares at the model's first iteration, else the entry of largest magnitude with the first index on ties (as
// idamax).  On the last mode also lambda_j * <F_j, G_j> for the error term.  grid = (column groups, slots).
constexpr int WIDE_STAT_COLS = 32;
__global__ void __launch_bounds__(WIDE_THREADS) wide_stats_kernel(const WideParams p) {
  const int m = wide_find_model(p, blockIdx.y);
  if (m < 0)
    return;
  const ModelDesc &md = p.models[m];
  const int R = md.rank, rows = p.rows, ld = p.ld, iters = md.iters;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const WideSlot w = wide_slot(p, blockIdx.y);
  double *Fm = wide_factor(p) + (size_t)md.col * ld;
  const double *Gm = p.G + (size_t)md.col * ld;
  const bool jk_here = md.jk_mode == p.mode, last_mode = p.mode == p.n_modes - 1;
#pragma unroll 1
  for (int j = blockIdx.x * WIDE_STAT_COLS + warp; j < min(R, (int)(blockIdx.x + 1) * WIDE_STAT_COLS); j += 8) {
    double *fj = Fm + (size_t)j * ld;
    if (jk_here && lane == 0)
      fj[md.jk_fiber] *= 0.0;
    __syncwarp();
    double lam;
    if (iters == 1) {
      double ss = 0.0;
      for (int r = lane; r < rows; r += 32)
        ss += fj[r] * fj[r];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1)
        ss += __shfl_xor_sync(0xffffffffu, ss, o);
      lam = sqrt(ss);
    } else {
      double best = -1.0;
      int bi = 0x7fffffff;
      for (int r = lane; r < rows; r += 32) {
        const double a = fabs(fj[r]);
        if (a > best) { // strictly greater keeps the first index of this lane's rows
          best = a;
          bi = r;
        }
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
      lam = fj[bi == 0x7fffffff ? 0 : bi];
    }
    const double rl = (lam != 0.0) ? 1.0 / lam : 1.0;
    __syncwarp();
    double t3 = 0.0;
    for (int r = lane; r < rows; r += 32) {
      const double v = fj[r] * rl;
      fj[r] = v;
      if (last_mode)
        t3 += lam * v * Gm[(size_t)j * ld + r];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
      t3 += __shfl_xor_sync(0xffffffffu, t3, o);
    if (lane == 0) {
      p.lambda_home[md.home_col + j] = lam;
      w.lam[j] = lam;
      w.t3[j] = t3;
    }
  }
}

// Gram_n = F^T F: CTA t of a slot computes tile t of the lower block triangle over all rows and writes it and its mirror
// image.  grid = (tiles of the largest wide model, slots).
__global__ void __launch_bounds__(WIDE_THREADS, 2) wide_gram_kernel(const WideParams p) {
  const int m = wide_find_model(p, blockIdx.y);
  if (m < 0)
    return;
  const ModelDesc &md = p.models[m];
  const int R = md.rank, NT = (R + WIDE_NB - 1) / WIDE_NB, ld = p.ld;
  const int t = blockIdx.x;
  if (t >= NT * (NT + 1) / 2)
    return;
  int ti = 0;
  while ((ti + 1) * (ti + 2) / 2 <= t)
    ti++;
  const int tj = t - ti * (ti + 1) / 2;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const double *Fm = wide_factor(p) + (size_t)md.col * ld;
  extern __shared__ double wsm[];
  double *sA = wsm, *sB = sA + WIDE_TILE;
  double acc[8][2];
  wide_acc_zero(acc);
#pragma unroll 1
  for (int r0 = 0; r0 < p.rows; r0 += WIDE_NB) {
    __syncthreads();
    wide_stage(sA, Fm, ld, r0, ti * WIDE_NB, p.rows, R);
    wide_stage(sB, Fm, ld, r0, tj * WIDE_NB, p.rows, R);
    __syncthreads();
    wide_tile_mma<true, false>(acc, sA, sB, warp, lane); // C(i, j) = sum_r F[r][i] F[r][j]
  }
  double *g = p.gram_pool + md.gram_off + (size_t)p.mode * R * R;
  const int r = lane >> 2, s = lane & 3, i = ti * WIDE_NB + 8 * warp + r;
  if (i >= R)
    return;
#pragma unroll
  for (int jj = 0; jj < 8; jj++)
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int j = tj * WIDE_NB + 8 * jj + 2 * s + h;
      if (j < R && (ti != tj || j <= i)) { // a diagonal tile contributes its lower triangle to both halves
        g[i + (size_t)j * R] = acc[jj][h];
        g[j + (size_t)i * R] = acc[jj][h];
      }
    }
}

// Last mode: fast error (reference src/utils/error.cpp:64-89), fit and the eviction decision.  grid = slots.
__global__ void __launch_bounds__(WIDE_THREADS) wide_error_kernel(const WideParams p) {
  const int m = wide_find_model(p, blockIdx.x);
  if (m < 0)
    return;
  ModelDesc &md = p.models[m];
  SchedState *st = p.st;
  const int R = md.rank, tid = threadIdx.x;
  const WideSlot w = wide_slot(p, blockIdx.x);
  const double *gn = p.gram_pool + md.gram_off + (size_t)p.mode * R * R;
  __shared__ double red[32];
  double term2 = 0.0, term3 = 0.0;
  for (int e = tid; e < R * R; e += WIDE_THREADS) {
    const int i = e % R, j = e / R;
    term2 += w.lam[i] * w.lam[j] * w.H[i + (size_t)j * p.ldw] * gn[e];
  }
  for (int j = tid; j < R; j += WIDE_THREADS)
    term3 += w.t3[j];
  term2 = block_sum(term2, red);
  term3 = block_sum(term3, red);
  if (tid == 0) {
    double xn = st->x_norm;
    if (md.jk_mode >= 0 && p.x_norms_jk)
      xn = p.x_norms_jk[md.jk_fiber];
    const double err = sqrt(fmax(xn * xn + term2 - 2.0 * term3, 0.0));
    md.error = err;
    md.old_fit = md.fit;
    md.fit = 1.0 - fabs(err) / st->x_norm;
    if (!st->ls_enabled) // with line search the decision is taken after the extrapolation step (ls.cuh)
      decide_eviction(md, st);
  }
}

} // namespace calsb200
