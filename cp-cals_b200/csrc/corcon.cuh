// Core consistency diagnostic (CORCONDIA; Bro & Kiers, J. Chemometrics 17 (2003) 274-286; corcond.m of the N-way
// toolbox) of every queued model, 3 and 4 modes.  For a model with factors F_n and weights lambda, A_0 = F_0 diag(lambda),
// A_n = F_n (n >= 1):
//
//   P_n = A_n (A_n^T A_n)^-1                           corcon_pinv_kernel: one CTA per (model, mode)
//   T   = X x_0 P_0   (all columns of a batch at once) pair_gemm_kernel (pairnode.cuh), unchanged, on a 3-D view
//                                                      (I_0, I_1, prod_{n>=2} I_n) of the tensor
//   G   = T x_1 P_1 x_2 P_2 (x_3 P_3)                  corcon_chain_kernel, one launch per mode for the whole batch
//   CC  = 100 (1 - sum (G - I)^2 / R)                  corcon_final_kernel: one CTA per model
//
// G is the least-squares Tucker core of X with the model's factors as Tucker bases.  A jackknife sub-model leaves out
// row jk_fiber of mode 0: that row of A_0 is zero, so P_0 has a zero row and the result is the core consistency of the
// row-deleted problem.  Every reduction runs in a fixed order (no atomics), and no product depends on which other
// models share a batch, so results are bit-identical from call to call and across batch sizes.
#pragma once
#include "update.cuh"

namespace calsb200 {

constexpr int CC_THREADS = 256;
constexpr int CC_FINAL_THREADS = 1024;
// A pivot d_j of the Cholesky factorisation of A^T A at or below CC_PIVOT_TOL * (A^T A)_jj counts as non-positive:
// rounding leaves the pivot of an exactly singular Gram matrix (two equal columns) a few ulps either side of zero.
constexpr double CC_PIVOT_TOL = 1e-12;
// 4 modes: the core has R^4 entries, 16.8 M at rank 64
constexpr int CC_MAX_RANK_4 = 64;

// One model of a batch.
struct CcModel {
  int model;    // queue position: index of the outputs and of the failure flags
  int rank;
  int home_col; // first column in the factor source and in lambda
  int bcol;     // first column in the batch's P_n and T
  int jk_row;   // mode-0 row left out (jackknife sub-model), -1: none
};

// One model's share of one contraction step: out(m, r) = sum_k in(k, m) P(k, r), in K x M (ld K), out M x R (ld M).
struct CcJob {
  long long in_off, out_off; // doubles into the step's input / output buffer
  long long M;
  long long tile0; // first CTA of this model in the step's grid (CC_CHAIN_MT rows of out per CTA)
  int R, bcol;
};

struct CcPinvParams {
  int n_modes;
  int dims[CALS_MAX_MODES];
  int ld[CALS_MAX_MODES];     // pitch of F and P (I_n rounded up to even)
  const double *F[CALS_MAX_MODES]; // factor source: home matrices after a run, else the uploaded queue
  const double *lambda;       // per source column; nullptr: all ones
  double *P[CALS_MAX_MODES];  // ld x batch columns
  const CcModel *models;
  int *fail;                  // [model * n_modes + mode]: 1 when A_n^T A_n is not numerically positive definite
  int max_rows;               // longest mode
};

// Shared memory of corcon_pinv_kernel: two LD x LD matrices, two LD vectors, the staged chunk (pitch x LD).
__host__ __device__ inline size_t cc_pinv_smem(int R, int pitch) {
  const size_t LD = (size_t)((R + 7) & ~7);
  return (2 * LD * LD + 2 * LD + (size_t)pitch * LD) * 8;
}

// Rows of A_n that corcon_pinv_kernel stages at a time for a rank-R model: as many as CC_PINV_SMEM_BUDGET allows, at
// most the longest mode (a multiple of 32; the pitch of the chunk is 4 more, 4 mod 16 doubles).  It depends on R alone
// because the Gram matrix is summed chunk by chunk: a model's result must not depend on the other models of its batch.
constexpr size_t CC_PINV_SMEM_BUDGET = 200 * 1024;
__host__ __device__ inline int cc_chunk_rows(int R, int max_rows) {
  int cr = (max_rows + 31) / 32 * 32;
  while (cr > 32 && cc_pinv_smem(R, cr + 4) > CC_PINV_SMEM_BUDGET)
    cr -= 32;
  return cr;
}

// P_n = A_n (A_n^T A_n)^-1 from the building blocks of model_update_kernel (update.cuh): Gram matrix by gram_dmma over
// staged row chunks, Cholesky by one warp, inverses of L's 8 x 8 diagonal blocks, and the blocked DMMA solve of every
// row against L L^T.  A failed factorisation writes P_n = 0 (the model's columns of T stay finite) and raises the flag.
__global__ void __launch_bounds__(CC_THREADS) corcon_pinv_kernel(const CcPinvParams p) {
  const CcModel md = p.models[blockIdx.x];
  const int n = blockIdx.y, N = p.n_modes;
  const int R = md.rank, LD = (R + 7) & ~7;
  const int rows = p.dims[n], ld = p.ld[n];
  const int tid = threadIdx.x, nthr = blockDim.x, warp = tid >> 5, lane = tid & 31, nw = nthr >> 5;
  const int CR = cc_chunk_rows(R, p.max_rows), pitch = CR + 4;
  extern __shared__ double sm[];
  double *Hs = sm;            // LD x LD: A^T A (lower block triangle), then L in its lower triangle
  double *Di = Hs + LD * LD;  // LD x LD: inverses of L's diagonal blocks, zero elsewhere
  double *inv = Di + LD * LD; // LD: 1 / L[j][j]
  double *hdiag = inv + LD;   // LD: diagonal of A^T A
  double *S = hdiag + LD;     // staged rows, column-major, pitch x LD
  __shared__ int s_fail;
  const double *F = p.F[n] + (size_t)md.home_col * ld;
  const double *lam = (n == 0 && p.lambda != nullptr) ? p.lambda + md.home_col : nullptr;
  const int skip_row = n == 0 ? md.jk_row : -1;
  double *Pm = p.P[n] + (size_t)md.bcol * ld;

  for (int e = tid; e < 2 * LD * LD + 2 * LD; e += nthr)
    sm[e] = 0.0;
  // rows [r0, r0 + nr) of A_n into S; columns R .. LD-1 zero (the tensor-core loops read them)
  auto stage = [&](int r0, int nr) {
#pragma unroll 1
    for (int j = warp; j < LD; j += nw) {
      double *sj = S + (size_t)j * pitch;
      if (j < R) {
        const double *fj = F + (size_t)j * ld + r0;
        const double sc = lam ? lam[j] : 1.0;
        for (int rr = lane; rr < nr; rr += 32)
          sj[rr] = (r0 + rr == skip_row) ? 0.0 : fj[rr] * sc;
      } else
        for (int rr = lane; rr < nr; rr += 32)
          sj[rr] = 0.0;
    }
  };
  __syncthreads();

  // ---- A^T A ----
#pragma unroll 1
  for (int r0 = 0; r0 < rows; r0 += CR) {
    const int nr = min(CR, rows - r0);
    stage(r0, nr);
    __syncthreads();
    gram_dmma(S, pitch, nr, Hs, LD, warp, nw, lane);
    __syncthreads();
  }

  // ---- L L^T = A^T A, block inverses ----
  if (warp == 0) {
    for (int j = lane; j < R; j += 32)
      hdiag[j] = Hs[j + j * LD];
    __syncwarp();
    int fail = cholesky_warp(Hs, LD, inv, R, lane);
    for (int j = lane; j < R; j += 32) {
      const double l = Hs[j + j * LD];
      if (!(l * l > CC_PIVOT_TOL * hdiag[j]))
        fail = 1;
    }
    fail = __any_sync(0xffffffffu, fail);
    diag_block_inverses_warp(Hs, LD, inv, Di, R, lane);
    if (lane == 0)
      s_fail = fail;
  }
  __syncthreads();
  const bool failed = s_fail != 0;
  if (tid == 0)
    p.fail[(size_t)md.model * N + n] = failed ? 1 : 0;
  if (failed) {
    for (int j = warp; j < R; j += nw)
      for (int r = lane; r < rows; r += 32)
        Pm[(size_t)j * ld + r] = 0.0;
    return;
  }

  // ---- P = A (L L^T)^-1, row chunk by row chunk ----
#pragma unroll 1
  for (int r0 = 0; r0 < rows; r0 += CR) {
    const int nr = min(CR, rows - r0);
    if (r0 > 0)
      __syncthreads(); // S is free again
    stage(r0, nr);
    __syncthreads();
    solve_rows_dmma(S, pitch, nr, Hs, Di, LD, warp, nw, lane);
    __syncthreads();
#pragma unroll 1
    for (int j = warp; j < R; j += nw)
      for (int rr = lane; rr < nr; rr += 32)
        Pm[(size_t)j * ld + r0 + rr] = S[(size_t)j * pitch + rr];
  }
}

// One contraction step of the per-model chain for every model of a batch: out(m, r) = sum_k in(k, m) P(k, r), a batched
// A^T B product with K contiguous in both operands.  The output is written with r slowest, so the next step contracts
// the leading index again.  A CTA computes CC_CHAIN_MT rows of one model's output and all of its R (<= 96) columns:
// warp w owns m8 row group w and the R/8 n8 groups.  K runs through shared memory in chunks of CC_CHAIN_KC; the staged
// tiles are zero-padded (rows beyond M, columns beyond R, k beyond K), so the DMMA loop carries no masks.  The k order
// of every output element is fixed by K alone.
constexpr int CC_CHAIN_MT = 64;
constexpr int CC_CHAIN_KC = 32;
constexpr int CC_CHAIN_PITCH = CC_CHAIN_KC + 4; // 4 mod 16 doubles: the fragment loads are bank-conflict free
constexpr int CC_CHAIN_NB = 12;                 // n8 groups: R <= 96
__global__ void __launch_bounds__(CC_THREADS) corcon_chain_kernel(const CcJob *__restrict__ jobs, int n_jobs, int K,
                                                                  const double *__restrict__ in,
                                                                  const double *__restrict__ P, int ldP,
                                                                  double *__restrict__ out) {
  __shared__ __align__(16) double As[CC_CHAIN_MT * CC_CHAIN_PITCH];
  __shared__ __align__(16) double Bs[8 * CC_CHAIN_NB * CC_CHAIN_PITCH];
  int lo = 0, hi = n_jobs - 1; // the model whose tiles hold this CTA: last job with tile0 <= blockIdx.x
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (jobs[mid].tile0 <= (long long)blockIdx.x)
      lo = mid;
    else
      hi = mid - 1;
  }
  const CcJob jb = jobs[lo];
  const long long m0 = ((long long)blockIdx.x - jb.tile0) * CC_CHAIN_MT, M = jb.M;
  const int R = jb.R, NB = (R + 7) >> 3;
  const double *A = in + jb.in_off;
  const double *B = P + (size_t)jb.bcol * ldP;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, r = lane >> 2, s = lane & 3;
  double acc[CC_CHAIN_NB][2];
#pragma unroll
  for (int j = 0; j < CC_CHAIN_NB; j++)
    acc[j][0] = acc[j][1] = 0.0;
#pragma unroll 1
  for (int k0 = 0; k0 < K; k0 += CC_CHAIN_KC) {
    __syncthreads(); // the previous chunk has been read
    for (int e = tid; e < CC_CHAIN_MT * CC_CHAIN_KC; e += CC_THREADS) {
      const int kk = e % CC_CHAIN_KC, mm = e / CC_CHAIN_KC, k = k0 + kk;
      const long long m = m0 + mm;
      As[mm * CC_CHAIN_PITCH + kk] = (m < M && k < K) ? A[m * K + k] : 0.0;
    }
    for (int e = tid; e < 8 * NB * CC_CHAIN_KC; e += CC_THREADS) {
      const int kk = e % CC_CHAIN_KC, nn = e / CC_CHAIN_KC, k = k0 + kk;
      Bs[nn * CC_CHAIN_PITCH + kk] = (nn < R && k < K) ? B[(size_t)nn * ldP + k] : 0.0;
    }
    __syncthreads();
    const int kend = (min(CC_CHAIN_KC, K - k0) + 3) & ~3;
    const double *a = As + (8 * warp + r) * CC_CHAIN_PITCH + s;
    const double *b = Bs + r * CC_CHAIN_PITCH + s;
#pragma unroll 2
    for (int kk = 0; kk < kend; kk += 4) {
      const double av = a[kk];
#pragma unroll
      for (int j = 0; j < CC_CHAIN_NB; j++)
        if (j < NB)
          dmma_m8n8k4(acc[j][0], acc[j][1], av, b[8 * j * CC_CHAIN_PITCH + kk]);
    }
  }
  const long long row = m0 + 8 * warp + r;
  if (row >= M)
    return;
  double *o = out + jb.out_off + row;
#pragma unroll
  for (int j = 0; j < CC_CHAIN_NB; j++) {
    const int col = 8 * j + 2 * s;
    if (j < NB && col < R)
      o[(size_t)col * M] = acc[j][0];
    if (j < NB && col + 1 < R)
      o[(size_t)(col + 1) * M] = acc[j][1];
  }
}

// CC = 100 (1 - sum (G - I)^2 / R) per model; G = R^N entries, index r_0 + R r_1 + R^2 r_2 (+ R^3 r_3).  Every thread
// sums a fixed stride of entries, block_sum adds the partial sums in a fixed tree.
__global__ void __launch_bounds__(CC_FINAL_THREADS) corcon_final_kernel(const CcModel *__restrict__ models,
                                                                        const CcJob *__restrict__ last, int n_modes,
                                                                        const double *__restrict__ Gbuf,
                                                                        const int *__restrict__ fail,
                                                                        double *__restrict__ cc, int *__restrict__ status) {
  __shared__ double red[32];
  const CcModel md = models[blockIdx.x];
  const int R = md.rank;
  long long size = 1, dstep = 0; // R^N entries; the superdiagonal steps by 1 + R + .. + R^(N-1)
  for (int k = 0; k < n_modes; k++) {
    dstep += size;
    size *= R;
  }
  const double *G = Gbuf + last[blockIdx.x].out_off;
  double acc = 0.0;
  for (long long e = threadIdx.x; e < size; e += blockDim.x) {
    const double v = G[e] - (e % dstep == 0 ? 1.0 : 0.0);
    acc += v * v;
  }
  const double ss = block_sum(acc, red);
  if (threadIdx.x == 0) {
    int bad = 0;
    for (int k = 0; k < n_modes; k++)
      bad |= fail[(size_t)md.model * n_modes + k];
    status[md.model] = bad ? 2 : 0;
    cc[md.model] = bad ? __longlong_as_double(0x7ff8000000000000ll) : 100.0 * (1.0 - ss / (double)R);
  }
}

} // namespace calsb200
