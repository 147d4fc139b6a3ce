// Concurrent MTTKRP for sm_100a.
//
// Replaces mttkrp::mttkrp / mttkrp_impl / khatri_rao* / mttkrp_twostep* (reference src/utils/mttkrp.cpp:78-614) and the
// cuBLAS + khatri_rao_cuda path (src/utils/khatri_rao.cu:10-55):
//     G[i_n, c] = sum_{i_k, k != n} X[i_0 .. i_{N-1}] * prod_{k != n} A_k[i_k, c]        for all C live columns.
//
// Formulation (fused two-step contraction, Khatri-Rao product never materialised):
//   view X as (P, M, O): P = the memory-contiguous mode p (mode 0, or mode 1 of the mode-swapped copy when n == 0),
//   M = mode n, O = all remaining "outer" modes.  Then
//     G[m, c] = sum_o  w_o[c] * ( sum_p X[p, m, o] * A_p[p, c] ),     w_o[c] = prod_{outer k} A_k[i_k(o), c]
//   The inner sum is an FP64 tensor-core contraction (mma.sync m8n8k4 -> DMMA.8x8x4): the A_p tile stays resident in
//   shared memory for a whole sweep over o, X tiles stream through a TMA + mbarrier ring, and the outer scaling w_o[c]
//   is applied to the B fragments in registers, so the KRP row (p,o) is formed on the fly and never stored.
//
// Parallelisation: stream-K.  The (m-tile, n-tile, K-chunk) space is flattened and cut into gridDim.x equal contiguous
// ranges; each CTA writes one partial tile per (m,n) pair it touches into a workspace and mttkrp_reduce_kernel sums
// the partials in a fixed order (deterministic, no atomics).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include "common.cuh"

namespace calsb200 {

// ------------------------------------------------------------------------------------------------------------------
// Tile configuration.  K tile = 40 doubles: a dense [rows][40] shared-memory tile has a row pitch of 320 B = 8 mod 16
// doubles, which makes the paired-k LDS.128 fragment loads below bank-conflict free without padding or swizzle.
constexpr int KT = 40;           // K tile along the contiguous mode (multiple of 8, == 8 mod 16)
constexpr int OC = 8;            // outer indices per w-chunk
constexpr int NUM_MMA_WARPS = 8;
constexpr int NUM_PRODUCER_WARPS = 4; // a whole warpgroup, so that setmaxnreg can hand its registers to the MMA warps
constexpr int MTTKRP_THREADS = (NUM_MMA_WARPS + NUM_PRODUCER_WARPS) * 32;
constexpr int X_STAGES = 4;

template <int WM, int WN> struct TileCfg {
  static constexpr int M_TILE = 8 * WM;
  static constexpr int N_TILE = 8 * WN * NUM_MMA_WARPS;
  static constexpr int X_STAGE_BYTES = M_TILE * KT * 8;
  static constexpr int B_BYTES = N_TILE * KT * 8;
  static constexpr int W_BYTES = N_TILE * OC * 8;
  static constexpr int SMEM_BYTES = B_BYTES + X_STAGES * X_STAGE_BYTES + 2 * W_BYTES + 256;
};

struct MttkrpGeom {
  int mode;    // n
  int In;      // extent of mode n (rows of G)
  int Ip;      // extent of the contiguous mode p
  int p_mode;
  int n_outer;
  int outer_mode[CALS_MAX_OUTER]; // ascending; [0] is the fastest outer mode q
  int outer_dim[CALS_MAX_OUTER];
  int outer_lmul[CALS_MAX_OUTER]; // contribution of the outer index to TMA coordinate 1 (modes between p and n)
  int outer_umul[CALS_MAX_OUTER]; // contribution to TMA coordinate 3 (modes above n)
  int P_tiles; // ceil(Ip / KT)
  int QC;      // ceil(outer_dim[0] / OC)
  int S;       // prod(outer_dim[1..])
  int m_tiles; // ceil(In / M_TILE)
  int ldG;
  int ldF[CALS_MAX_MODES];
  // Slab mode (tensor sliced along one mode over several GPUs, BASELINE config 5): the tensor on this device covers
  // rows [off, off + extent) of the sliced mode's factor.  Offsets are 0 everywhere else.
  int outer_off[CALS_MAX_OUTER]; // row offset into the factor of every outer mode
  int g_row_off;                 // row offset of this device's G rows (non-zero only when mode == sliced mode)
  int carry_fallback; // runs only when SchedState::carry_ok is 0 (mode 0 in an odd pass of the multi-sweep schedule)
};

struct MttkrpMaps {
  CUtensorMap X;     // 4-D view (P, L', M, U) of the tensor copy used for this mode
  CUtensorMap B[2];  // factor p in buffer 0 / 1: 2-D (Ip, buffer_cols)
  CUtensorMap W[2];  // factor q (fastest outer mode) in buffer 0 / 1
  CUtensorMap Bn[2]; // the same two with a box of NARROW_COLS columns (narrow column tail)
  CUtensorMap Wn[2];
};

// Narrow column tail.  When the live column count C leaves at most NARROW_COLS columns in its last 64-column octet (and
// there is at least one full octet), those columns are not given a slot of the regular warp layout -- one n8 group per
// warp and octet, so a tail of 7 columns keeps one warp of eight busy for a whole octet slot and costs the tile its
// pipeline fill (measured: 263 columns ran 23 % slower than 255) -- but are computed by a second, NARROW instance of the
// contraction kernels in which the eight warps split the ROWS of the tile (warp w = m8 row group w) and every warp
// covers all of the tail's (at most four) n8 groups.  The main instances then see only full octets.
// Tuning knob (CALS_B200_NARROW=1), off by default: the second persistent kernel costs what it saves (engine.cu).
constexpr int NARROW_GROUPS = 4;
constexpr int NARROW_COLS = 8 * NARROW_GROUPS;
__host__ __device__ inline int narrow_cols(int C) {
  const int NO = (C + 63) >> 6, tail = C - 64 * (NO - 1);
  return (NO >= 2 && tail <= NARROW_COLS) ? tail : 0;
}

// ------------------------------------------------------------------------------------------------------------------
// PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  uint32_t done;
  const uint32_t addr = smem_u32(bar);
  do {
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done)
                 : "r"(addr), "r"(parity)
                 : "memory");
  } while (!done);
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_load_3d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_load_4d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
               ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void dmma_m8n8k4(double &c0, double &c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
      : "+d"(c0), "+d"(c1)
      : "d"(a), "d"(b));
}

// ------------------------------------------------------------------------------------------------------------------
// Work partition ("plan"): cost-weighted stream-K, computed on the device by the scheduler (sched.cuh) whenever the
// number of live columns changes, and read as tables by the MTTKRP and reduce kernels.
//
//   * G is split into m-tiles of at most WM m8 row groups (even split of ceil(In/8) groups, so tiles differ by at most
//     one group) and into n-tiles of at most 4 "octets" (octet = 8 n8 column groups = 64 columns, one n8 group per MMA
//     warp), again an even split.  Inside a tile, octet j / group w (columns 64*j + 8*w ..) belongs to warp w, so every
//     warp of a CTA has the same number nn of column groups and no per-warp predicates are needed; only the last octet
//     of the last tile can reach beyond C, where TMA zero-fills the factor tile.
//   * Every (m,n) pair has Tp stages (PlanShape below); a stage of pair (mt, nt) is priced by the DMMAs it issues,
//     groups * 2*nm(mt)*nn(nt), plus a fixed per-stage cost.  The flattened stage sequence is cut into
//     G_eff = min(G, #stages) contiguous ranges of (nearly) equal cost, every range non-empty.
//   * A "segment" is the part of one CTA's range that lies in one pair; segments are numbered globally in stage order
//     and segment s writes workspace tile s.  The segments of a pair are consecutive: the reduce kernel sums tiles
//     pair_seg0[pair] .. pair_seg0[pair+1]-1 in that order (deterministic, no atomics).
constexpr int N8_TILE = 32; // n8 groups per full n-tile (8 warps x WN = 4)
constexpr int OCT_TILE = 4; // octets per full n-tile
constexpr int PLAN_HDR = 8;

struct PlanView {
  int n_tiles, m_tiles, pairs, Tp, G_eff, n_segments, NO, In8; // NO = number of 64-column octets covering C
  const int *cta_lo;    // [G + 1]
  const int *cta_seg0;  // [G]
  const int *pair_seg0; // [pairs + 1]
};

__host__ __device__ inline int plan_capacity(int G, int pairs_max) { return PLAN_HDR + (G + 1) + G + (pairs_max + 1); }
__host__ __device__ inline int plan_wm(int mt, int In8, int m_tiles) {
  return (int)(((long long)(mt + 1) * In8) / m_tiles - ((long long)mt * In8) / m_tiles);
}
__host__ __device__ inline int plan_m8_start(int mt, int In8, int m_tiles) {
  return (int)(((long long)mt * In8) / m_tiles);
}
__host__ __device__ inline int plan_oct_start(int nt, int NO, int n_tiles) {
  return (int)(((long long)nt * NO) / n_tiles);
}
__host__ __device__ inline int plan_nn(int nt, int NO, int n_tiles) {
  return plan_oct_start(nt + 1, NO, n_tiles) - plan_oct_start(nt, NO, n_tiles);
}
// tile that holds item x under the even split of `count` items over `tiles` tiles (start(t) = floor(t*count/tiles))
__host__ __device__ inline int plan_tile_of(int x, int count, int tiles) {
  int t = (int)(((long long)(x + 1) * tiles - 1) / count);
  while ((int)(((long long)t * count) / tiles) > x)
    t--;
  while (t + 1 < tiles && (int)(((long long)(t + 1) * count) / tiles) <= x)
    t++;
  return t;
}
__host__ __device__ inline PlanView plan_view(const int *plan, int G) {
  PlanView v;
  v.n_tiles = plan[0];
  v.m_tiles = plan[1];
  v.pairs = plan[2];
  v.Tp = plan[3];
  v.G_eff = plan[4];
  v.n_segments = plan[5];
  v.NO = plan[6];
  v.In8 = plan[7];
  v.cta_lo = plan + PLAN_HDR;
  v.cta_seg0 = plan + PLAN_HDR + (G + 1);
  v.pair_seg0 = plan + PLAN_HDR + (G + 1) + G;
  return v;
}

// Shape of one mode's work space.  The unit of work is a STAGE: one X tile (K tile pt, slow outer index sl, fastest
// outer index iq), iq fastest; Tp = P_tiles * S * Iq stages per (m,n) pair.  Stages are grouped in chunks of OC
// consecutive iq (one weight-tile load per chunk); a CTA's range may begin and end inside a chunk.
struct PlanShape {
  int In, WM; // rows of G on this device, tallest m-tile in m8 groups
  int Ip;     // extent of the contiguous (K) mode  -> P_tiles = ceil(Ip / KT), the last tile may hold fewer K8 groups
  int Iq;     // extent of the fastest outer mode
  int S;      // product of the slower outer extents
};
__host__ __device__ inline int plan_p_tiles(const PlanShape &sh) { return (sh.Ip + KT - 1) / KT; }
__host__ __device__ inline long long plan_tp(const PlanShape &sh) {
  return (long long)plan_p_tiles(sh) * sh.S * sh.Iq;
}

// Cost model (unit: one DMMA issue slot of one warp): a stage costs groups * 2*nm*nn DMMAs plus PLAN_STAGE_COST of
// barrier / weight bookkeeping (the per-chunk weight-tile wait spread over its stages).  Stages of the last K tile hold
// ceil(tail / 8) groups instead of KT / 8 and are priced as such -- what an equal-weight split gets wrong on ragged
// shapes (299 x 301 x 41).
constexpr int PLAN_STAGE_COST = 5;
struct PairCost {
  long long stage_full, stage_tail; // cost of one stage in a full / in the last K tile
  long long full_stages;            // stages of the pair that lie in full K tiles
  __host__ __device__ long long prefix(long long k) const { // cost of the first k stages of the pair
    const long long nf = k < full_stages ? k : full_stages;
    return nf * stage_full + (k - nf) * stage_tail;
  }
};
// g_last: valid n8 groups in the pair's last octet (8 = full).  Warps g_last..7 skip that octet's slot; a sub-partition
// runs warps q and q + 4, so the busiest one (q = 0) issues nn + (g_last > 4 ? nn : nn - 1) slots per row group.
__host__ __device__ inline PairCost plan_pair_cost(const PlanShape &sh, int nm, int nn, int g_last = 8) {
  PairCost pc;
  const int P_tiles = plan_p_tiles(sh);
  const int tail_groups = (sh.Ip - (P_tiles - 1) * KT + 7) / 8;
  const long long per_group = (long long)nm * (nn + (g_last > 4 ? nn : nn - 1));
  pc.stage_full = (long long)(KT / 8) * per_group + PLAN_STAGE_COST;
  pc.stage_tail = (long long)tail_groups * per_group + PLAN_STAGE_COST;
  pc.full_stages = (long long)(P_tiles - 1) * sh.S * sh.Iq;
  return pc;
}

// Builds the plan for one mode.  O((G + pairs) * log Tp) integer steps, single thread.
__host__ __device__ inline void mttkrp_make_plan(int *plan, const PlanShape &sh, int C, int G) {
  const int In = sh.In, WM = sh.WM;
  const int Tp = (int)plan_tp(sh);
  const int In8 = (In + 7) / 8, NO = (C + 63) / 64;
  const int m_tiles = (In8 + WM - 1) / WM;
  const int n_tiles = (NO + OCT_TILE - 1) / OCT_TILE;
  const int pairs = m_tiles * n_tiles;
  const long long total = (long long)pairs * Tp;
  const int G_eff = (int)(total < (long long)G ? total : (long long)G);
  const int g_tail = (C - 64 * (NO - 1) + 7) / 8; // valid n8 groups of the very last octet (1..8)
  int *cta_lo = plan + PLAN_HDR, *cta_seg0 = plan + PLAN_HDR + (G + 1), *pair_seg0 = plan + PLAN_HDR + (G + 1) + G;
  // total weight
  long long W = 0;
  for (int pi = 0; pi < pairs; pi++) {
    const int nt = pi / m_tiles, mt = pi - nt * m_tiles;
    W += plan_pair_cost(sh, plan_wm(mt, In8, m_tiles), plan_nn(nt, NO, n_tiles), nt == n_tiles - 1 ? g_tail : 8)
             .prefix(Tp);
  }

  int pi = 0, k = 0, seg = 0;
  long long cw = 0, done = 0;
  PairCost pc = plan_pair_cost(sh, plan_wm(0, In8, m_tiles), plan_nn(0, NO, n_tiles), n_tiles == 1 ? g_tail : 8);
  for (int b = 0; b < G_eff; b++) {
    cta_lo[b] = (int)done;
    cta_seg0[b] = seg;
    const long long target = (b == G_eff - 1) ? W : W * (b + 1) / G_eff;
    const long long must_leave = G_eff - b - 1;
    long long taken = 0;
    while (pi < pairs) {
      const long long r = Tp - k;
      const long long avail = total - done - must_leave;
      const long long base = pc.prefix(k);
      long long want;
      if (cw + (pc.prefix(Tp) - base) <= target)
        want = r;
      else { // largest want with cw + cost(k .. k+want) <= target
        long long lo = 0, hi = r;
        while (lo < hi) {
          const long long mid = (lo + hi + 1) / 2;
          if (cw + (pc.prefix(k + mid) - base) <= target)
            lo = mid;
          else
            hi = mid - 1;
        }
        want = lo;
      }
      if (taken == 0 && want <= 0)
        want = 1;
      if (want > r)
        want = r;
      if (want > avail)
        want = avail;
      if (want <= 0)
        break;
      if (k == 0)
        pair_seg0[pi] = seg;
      seg++;
      cw += pc.prefix(k + want) - base;
      k += (int)want;
      done += want;
      taken += want;
      if (k == Tp) {
        pi++;
        k = 0;
        if (pi < pairs) {
          const int nt = pi / m_tiles, mt = pi - nt * m_tiles;
          pc = plan_pair_cost(sh, plan_wm(mt, In8, m_tiles), plan_nn(nt, NO, n_tiles), nt == n_tiles - 1 ? g_tail : 8);
        }
      } else
        break;
    }
  }
  for (int b = G_eff; b <= G; b++)
    cta_lo[b] = (int)total;
  for (int b = G_eff; b < G; b++)
    cta_seg0[b] = seg;
  pair_seg0[pairs] = seg;
  plan[0] = n_tiles;
  plan[1] = m_tiles;
  plan[2] = pairs;
  plan[3] = Tp;
  plan[4] = G_eff;
  plan[5] = seg;
  plan[6] = NO;
  plan[7] = In8;
}

// One thread per mode builds its plan (test hook path; the run loop plans inside sched_kernel).
struct PlanArgs {
  int n_modes;
  PlanShape shape[CALS_MAX_MODES];
  int *plan[CALS_MAX_MODES];
  int G;
  int *built_for; // [2 * CALS_MAX_MODES] column count each plan table was last built for (-1: never); device memory:
                  // [n] for plan[n], [CALS_MAX_MODES + n] for plan_narrow[n]
  int *plan_narrow[CALS_MAX_MODES]; // plan of the narrow column tail (one n-tile), nullptr when the run has none
};
__global__ void mttkrp_plan_kernel(const PlanArgs a, int C, int narrow_on) {
  const int n = threadIdx.x;
  if (n < a.n_modes && a.plan[n]) {
    const int tail = (narrow_on && a.plan_narrow[n]) ? narrow_cols(C) : 0;
    mttkrp_make_plan(a.plan[n], a.shape[n], C - tail, a.G);
    if (tail)
      mttkrp_make_plan(a.plan_narrow[n], a.shape[n], tail, a.G);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// One K8 group of one stage for one warp: NM valid m8 row groups x NN n8 column groups (both CTA-uniform, compile time).
// SCALE = false: plain contraction (no outer weight), used by the pair-node kernel (pairnode.cuh).
template <int WM, int WN, int NM, int NN, bool SCALE = true>
__device__ __forceinline__ void mma_group(double (&acc)[WM][WN][2], const double *__restrict__ Xt,
                                          const double *__restrict__ Bw, const double (&wv)[WN], int gk, int r, int s) {
  double2 b[NN];
#pragma unroll
  for (int j = 0; j < NN; j++) {
    b[j] = *reinterpret_cast<const double2 *>(Bw + (j * 64 + r) * KT + gk * 8 + 2 * s);
    if (SCALE) {
      b[j].x *= wv[j];
      b[j].y *= wv[j];
    }
  }
  // Row group by row group: k = 8*gk + 2s first, then k = 8*gk + 2s + 1; only one A fragment is live at a time.
#pragma unroll
  for (int i = 0; i < NM; i++) {
    const double2 a = *reinterpret_cast<const double2 *>(Xt + (i * 8 + r) * KT + gk * 8 + 2 * s);
#pragma unroll
    for (int j = 0; j < NN; j++)
      dmma_m8n8k4(acc[i][j][0], acc[i][j][1], a.x, b[j].x);
#pragma unroll
    for (int j = 0; j < NN; j++)
      dmma_m8n8k4(acc[i][j][0], acc[i][j][1], a.y, b[j].y);
  }
}

// All K8 groups of one stage for a compile-time (NM, NN).
template <int WM, int WN, int NM, int NN, bool SCALE = true>
__device__ __forceinline__ void mma_stage_nm(double (&acc)[WM][WN][2], const double *Xt, const double *Bw,
                                             const double (&wv)[WN], int ngroups, int r, int s) {
  if (NM == WM && NN == WN && ngroups == KT / 8) { // the common case: fully unrolled
#pragma unroll
    for (int gk = 0; gk < KT / 8; gk++)
      mma_group<WM, WN, NM, NN, SCALE>(acc, Xt, Bw, wv, gk, r, s);
  } else {
#pragma unroll 1
    for (int gk = 0; gk < ngroups; gk++) // K tail: rows of the K tile beyond Ip are zero-filled by TMA, skip them
      mma_group<WM, WN, NM, NN, SCALE>(acc, Xt, Bw, wv, gk, r, s);
  }
}

template <int WM, int WN, int NM, bool SCALE = true>
__device__ __forceinline__ void mma_stage_n(double (&acc)[WM][WN][2], const double *Xt, const double *Bw,
                                            const double (&wv)[WN], int ngroups, int r, int s, int nn) {
  static_assert(WN == 4, "dispatch below assumes 4 column groups per warp");
  switch (nn) {
  case 0: // this warp's only column group of the tile starts beyond C
    break;
  case 1:
    mma_stage_nm<WM, WN, NM, 1, SCALE>(acc, Xt, Bw, wv, ngroups, r, s);
    break;
  case 2:
    mma_stage_nm<WM, WN, NM, 2, SCALE>(acc, Xt, Bw, wv, ngroups, r, s);
    break;
  case 3:
    mma_stage_nm<WM, WN, NM, 3, SCALE>(acc, Xt, Bw, wv, ngroups, r, s);
    break;
  default:
    mma_stage_nm<WM, WN, NM, 4, SCALE>(acc, Xt, Bw, wv, ngroups, r, s);
    break;
  }
}

template <int WM, int WN, bool SCALE = true>
__device__ __forceinline__ void mma_stage(double (&acc)[WM][WN][2], const double *Xt, const double *Bw,
                                          const double (&wv)[WN], int ngroups, int r, int s, int nm, int nn) {
  static_assert(WM >= 1 && WM <= 8, "extend the dispatch below");
#define CALS_MMA_CASE(NMV)                                                                                             \
  case NMV:                                                                                                            \
    if (WM >= NMV)                                                                                                     \
      mma_stage_n<WM, WN, (WM >= NMV ? NMV : 1), SCALE>(acc, Xt, Bw, wv, ngroups, r, s, nn);                           \
    break;
  switch (nm) {
    CALS_MMA_CASE(1)
    CALS_MMA_CASE(2)
    CALS_MMA_CASE(3)
    CALS_MMA_CASE(4)
    CALS_MMA_CASE(5)
    CALS_MMA_CASE(6)
    CALS_MMA_CASE(7)
    CALS_MMA_CASE(8)
  default:
    break;
  }
#undef CALS_MMA_CASE
}

// One stage of the NARROW instances for one warp: the warp's own m8 row group (rows row8*8 .. +7 of the X tile) times
// the g <= NARROW_GROUPS n8 column groups of the tail.  acc[q] belongs to column group q.
template <bool SCALE>
__device__ __forceinline__ void mma_narrow_stage(double (&acc)[NARROW_GROUPS][2], const double *__restrict__ Xt,
                                                 const double *__restrict__ Bs, const double (&wv)[NARROW_GROUPS],
                                                 int ngroups, int r, int s, int row8, int g) {
  const double *xa = Xt + (row8 * 8 + r) * KT + 2 * s;
  const double *xb = Bs + r * KT + 2 * s;
#pragma unroll 1
  for (int gk = 0; gk < ngroups; gk++) {
    const double2 a = *reinterpret_cast<const double2 *>(xa + gk * 8);
#pragma unroll
    for (int q = 0; q < NARROW_GROUPS; q++)
      if (q < g) {
        double2 b = *reinterpret_cast<const double2 *>(xb + q * 8 * KT + gk * 8);
        if (SCALE) {
          b.x *= wv[q];
          b.y *= wv[q];
        }
        dmma_m8n8k4(acc[q][0], acc[q][1], a.x, b.x);
        dmma_m8n8k4(acc[q][0], acc[q][1], a.y, b.y);
      }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// The DMMA kernel.  384 threads: warps 0..7 consume (LDS + DMMA) with 232 registers each, warp 8 lane 0 produces (TMA);
// warps 9..11 only exist so that the producer warpgroup can release its registers (setmaxnreg) and exit at once.
// NARROW = false: columns [0, C_main) (C_override > 0: [0, C_override)).  NARROW = true: the narrow column tail
// [C_main, C) (C_override > 0: [C_lo_override, C_override)) with its own plan and workspace of M_TILE x NARROW_COLS tiles.
template <int WM, int WN, bool NARROW = false>
__global__ void __launch_bounds__(MTTKRP_THREADS, 1)
mttkrp_dmma_kernel(const __grid_constant__ MttkrpMaps maps, const MttkrpGeom g, const SchedState *__restrict__ st,
                   const FactorPtrs fac, const int *__restrict__ plan, double *__restrict__ ws, int C_override,
                   int C_lo_override) {
  using Cfg = TileCfg<WM, WN>;
  constexpr int M_TILE = Cfg::M_TILE, N_TILE = Cfg::N_TILE;
  static_assert(WN * NUM_MMA_WARPS == N8_TILE, "n-tile must hold N8_TILE n8 groups");
  static_assert(WN == NARROW_GROUPS, "the narrow instance keeps its accumulators in acc[0][0 .. WN)");

  // 1024-byte aligned dynamic shared memory (TMA destinations need 128 B); indexing the array directly keeps the
  // pointers in the shared address space (LDS instead of generic LD)
  extern __shared__ __align__(1024) unsigned char smem[];
  double *Bs = (double *)smem;                                            // [N_TILE][KT]
  double *Xs = (double *)(smem + Cfg::B_BYTES);                           // [X_STAGES][M_TILE][KT]
  double *Ws = (double *)(smem + Cfg::B_BYTES + X_STAGES * Cfg::X_STAGE_BYTES); // [2][N_TILE][OC]
  uint64_t *bars = (uint64_t *)(smem + Cfg::B_BYTES + X_STAGES * Cfg::X_STAGE_BYTES + 2 * Cfg::W_BYTES);
  uint64_t *full_x = bars, *empty_x = bars + X_STAGES;
  uint64_t *full_w = bars + 2 * X_STAGES, *empty_w = full_w + 2;
  uint64_t *full_b = empty_w + 2, *empty_b = full_b + 1;

  pdl_enter();
  const int C = C_override > 0 ? C_override : (NARROW ? st->C : st->C_main);
  const int c_lo = NARROW ? (C_override > 0 ? C_lo_override : st->C_main) : 0; // first column of the narrow tail
  const int cur = C_override > 0 ? 0 : st->cur;
  if (C - c_lo <= 0 || (g.carry_fallback && st->carry_ok))
    return;
  const PlanView pv = plan_view(plan, gridDim.x);
  const int lo = pv.cta_lo[blockIdx.x], hi = pv.cta_lo[blockIdx.x + 1];
  if (lo >= hi)
    return;
  const int Tp = pv.Tp, m_tiles = pv.m_tiles, n_tiles = pv.n_tiles;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef CALS_B200_POISON_SMEM
  { // debug aid: any read of shared memory that no TMA has written shows up as NaN in G
    double *all = (double *)smem;
    const int nd = (Cfg::B_BYTES + X_STAGES * Cfg::X_STAGE_BYTES + 2 * Cfg::W_BYTES) / 8;
    for (int i = threadIdx.x; i < nd; i += blockDim.x)
      all[i] = __longlong_as_double(0x7ff8000000000000ll);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
  }
#endif
  if (threadIdx.x == 0) {
    for (int i = 0; i < X_STAGES; i++) {
      mbar_init(&full_x[i], 1);
      mbar_init(&empty_x[i], NUM_MMA_WARPS);
    }
    for (int i = 0; i < 2; i++) {
      mbar_init(&full_w[i], 1);
      mbar_init(&empty_w[i], NUM_MMA_WARPS);
    }
    mbar_init(full_b, 1);
    mbar_init(empty_b, NUM_MMA_WARPS);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  const int Iq = g.outer_dim[0];

  if (warp >= NUM_MMA_WARPS) {
    // ===================================== producer =====================================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");
    if (warp != NUM_MMA_WARPS || lane != 0)
      return;
    const CUtensorMap *tmB = &maps.B[cur], *tmW = &maps.W[cur];
    int xs = 0, wsi = 0;
    uint32_t xph = 1, wph = 1; // ring "empty" barriers: the first pass over the ring does not block
    uint32_t bph = 0;          // empty_b: k-th reload waits for the k-th release by the consumers
    int prev_key = -1;
    for (int u = lo; u < hi;) {
      // decode the stage: pair, K tile, slow outer index, fastest outer index
      const int pair = u / Tp;
      int lu = u - pair * Tp;
      const int nt = pair / m_tiles, mt = pair - nt * m_tiles;
      const int iq0 = lu % Iq;
      lu /= Iq;
      const int sl = lu % g.S, pt = lu / g.S;
      const int qc = iq0 / OC;
      // stages of this chunk that belong to this CTA: up to the end of the chunk, of the iq run, of the CTA's range
      const int n_here = min(min(OC - (iq0 - qc * OC), Iq - iq0), hi - u);
      const int key = pt * n_tiles + nt;
      if (key != prev_key) {
        if (prev_key >= 0) { // wait until all consumer warps have released the previous A_p tile
          mbar_wait(empty_b, bph);
          bph ^= 1;
        }
        if (NARROW) {
          mbar_expect_tx(full_b, NARROW_COLS * KT * 8);
          tma_load_2d(Bs, &maps.Bn[cur], full_b, pt * KT, c_lo);
        } else {
          mbar_expect_tx(full_b, Cfg::B_BYTES);
          tma_load_2d(Bs, tmB, full_b, pt * KT, 64 * plan_oct_start(nt, pv.NO, n_tiles));
        }
        prev_key = key;
      }
      // w chunk
      mbar_wait(&empty_w[wsi], wph);
      if (NARROW) {
        mbar_expect_tx(&full_w[wsi], NARROW_COLS * OC * 8);
        tma_load_2d(Ws + wsi * (N_TILE * OC), &maps.Wn[cur], &full_w[wsi], qc * OC, c_lo);
      } else {
        mbar_expect_tx(&full_w[wsi], Cfg::W_BYTES);
        tma_load_2d(Ws + wsi * (N_TILE * OC), tmW, &full_w[wsi], qc * OC, 64 * plan_oct_start(nt, pv.NO, n_tiles));
      }
      if (++wsi == 2) {
        wsi = 0;
        wph ^= 1;
      }
      // slow outer coordinates
      int lbase = 0, ubase = 0;
      {
        int rem = sl;
        for (int k = 1; k < g.n_outer; k++) {
          const int ik = rem % g.outer_dim[k];
          rem /= g.outer_dim[k];
          lbase += ik * g.outer_lmul[k];
          ubase += ik * g.outer_umul[k];
        }
      }
      const int m0 = 8 * plan_m8_start(mt, pv.In8, m_tiles);
      for (int o = 0; o < n_here; o++) {
        const int iq = iq0 + o;
        mbar_wait(&empty_x[xs], xph);
        mbar_expect_tx(&full_x[xs], Cfg::X_STAGE_BYTES);
        tma_load_4d(Xs + xs * (M_TILE * KT), &maps.X, &full_x[xs], pt * KT, lbase + iq * g.outer_lmul[0], m0,
                    ubase + iq * g.outer_umul[0]);
        if (++xs == X_STAGES) {
          xs = 0;
          xph ^= 1;
        }
      }
      u += n_here;
    }
    return;
  }

  // ===================================== consumers =====================================
  asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
  const int r = lane >> 2, s = lane & 3;
  // n8 group j*8 + warp of the n-tile belongs to this warp: column offset (j*8 + warp)*8 inside the tile
  const double *Bw = Bs + warp * 8 * KT;
  double acc[WM][WN][2];
#pragma unroll
  for (int i = 0; i < WM; i++)
#pragma unroll
    for (int j = 0; j < WN; j++)
      acc[i][j][0] = acc[i][j][1] = 0.0;
  double wslow[WN];
#pragma unroll
  for (int j = 0; j < WN; j++)
    wslow[j] = 1.0;

  int xs = 0, wsi = 0;
  uint32_t xph = 0, wph = 0, bph = 0;
  int prev_key = -1, prev_pair = -1, prev_sl = -1, prev_nt = -1;
  int seg = pv.cta_seg0[blockIdx.x] - 1;

  auto flush = [&]() {
    if (NARROW) { // warp = m8 row group, acc[0][q] = n8 column group q of the tail; tiles are M_TILE x NARROW_COLS
      double *tile = ws + (size_t)seg * (M_TILE * NARROW_COLS);
#pragma unroll
      for (int q = 0; q < NARROW_GROUPS; q++) {
        if (warp < WM)
          *reinterpret_cast<double2 *>(tile + (warp * 8 + r) * NARROW_COLS + q * 8 + 2 * s) =
              make_double2(acc[0][q][0], acc[0][q][1]);
        acc[0][q][0] = acc[0][q][1] = 0.0;
      }
      return;
    }
    double *tile = ws + (size_t)seg * (M_TILE * N_TILE);
#pragma unroll
    for (int i = 0; i < WM; i++)
#pragma unroll
      for (int j = 0; j < WN; j++) {
        double2 v = make_double2(acc[i][j][0], acc[i][j][1]);
        *reinterpret_cast<double2 *>(tile + (i * 8 + r) * N_TILE + (j * 8 + warp) * 8 + 2 * s) = v;
        acc[i][j][0] = acc[i][j][1] = 0.0;
      }
  };
  const int g_tail = NARROW ? min(NARROW_GROUPS, (C - c_lo + 7) >> 3) : 0; // n8 groups of the narrow tail

  for (int u = lo; u < hi;) {
    const int pair = u / Tp;
    int lu = u - pair * Tp;
    const int nt = pair / m_tiles, mt = pair - nt * m_tiles;
    const int iq0 = lu % Iq;
    lu /= Iq;
    const int sl = lu % g.S, pt = lu / g.S;
    const int qc = iq0 / OC, o0 = iq0 - qc * OC;
    const int n_here = min(min(OC - o0, Iq - iq0), hi - u); // same split of the range into chunk pieces as the producer
    // number of valid m8 row groups / n8 column groups of this pair (CTA-uniform)
    const int nm = plan_wm(mt, pv.In8, m_tiles);
    int nn = plan_nn(nt, pv.NO, n_tiles);
    // Only the last octet of the last n-tile can reach beyond C.  A warp whose n8 group of that octet starts at or beyond
    // C would multiply TMA zero-fill for a whole octet slot: it runs one slot less instead (per-warp, the barriers do not
    // depend on it).  C = 263 then costs 9 instead of 10 slots per SM sub-partition -- what the per-GPU shards of a
    // strong-scaled model set need; full octets are untouched.
    if (!NARROW && 64 * (plan_oct_start(nt, pv.NO, n_tiles) + nn - 1) + 8 * warp >= C)
      nn--;
    if (pair != prev_pair) {
      if (prev_pair >= 0)
        flush();
      seg++;
      prev_pair = pair;
    }
    const int key = pt * n_tiles + nt;
    if (key != prev_key) {
      if (prev_key >= 0) { // this warp is done with the previous A_p tile
        __syncwarp();
        if (lane == 0)
          mbar_arrive(empty_b);
      }
      mbar_wait(full_b, bph);
      bph ^= 1;
      prev_key = key;
    }
    if (g.n_outer > 1 && (sl != prev_sl || nt != prev_nt)) {
      // product of the slower outer factors for this thread's columns (rare: once per sweep of the fastest outer mode)
      int idx[CALS_MAX_OUTER];
      int rem = sl;
      for (int k = 1; k < g.n_outer; k++) {
        idx[k] = rem % g.outer_dim[k];
        rem /= g.outer_dim[k];
      }
#pragma unroll
      for (int j = 0; j < WN; j++) {
        // regular layout: n8 group (octet j, warp); narrow instance: n8 group j of the tail
        const int c = NARROW ? c_lo + j * 8 + r : 64 * plan_oct_start(nt, pv.NO, n_tiles) + (j * 8 + warp) * 8 + r;
        double w = 1.0;
        if (c < C)
          for (int k = 1; k < g.n_outer; k++) {
            const int md = g.outer_mode[k];
            w *= __ldg(fac.buf[cur][md] + (size_t)c * g.ldF[md] + idx[k] + g.outer_off[k]);
          }
        wslow[j] = w;
      }
    }
    prev_sl = sl;
    prev_nt = nt;

    mbar_wait(&full_w[wsi], wph);
    const double *Wc = Ws + wsi * (N_TILE * OC) + (NARROW ? 0 : warp * 8 * OC);
    const int kvalid = min(KT, g.Ip - pt * KT);
    const int ngroups = (kvalid + 7) >> 3;
    for (int o = o0; o < o0 + n_here; o++) {
      double wv[WN];
#pragma unroll
      for (int j = 0; j < WN; j++)
        wv[j] = Wc[((NARROW ? j * 8 : j * 64) + r) * OC + o] * wslow[j];
      mbar_wait(&full_x[xs], xph);
      if (NARROW) {
        if (warp < nm)
          mma_narrow_stage<true>(acc[0], Xs + xs * (M_TILE * KT), Bs, wv, ngroups, r, s, warp, g_tail);
      } else
        mma_stage<WM, WN>(acc, Xs + xs * (M_TILE * KT), Bw, wv, ngroups, r, s, nm, nn);
      __syncwarp();
      if (lane == 0)
        mbar_arrive(&empty_x[xs]);
      if (++xs == X_STAGES) {
        xs = 0;
        xph ^= 1;
      }
    }
    __syncwarp();
    if (lane == 0)
      mbar_arrive(&empty_w[wsi]);
    if (++wsi == 2) {
      wsi = 0;
      wph ^= 1;
    }
    u += n_here;
  }
  flush();
}

// ------------------------------------------------------------------------------------------------------------------
// Sum the partial tiles of every (m,n) pair in segment order and write G (In x C, column-major, ld = ldG).
// One CTA per 8 x 32 (rows x columns) patch of G, one output element per thread: reads are coalesced along columns of
// the row-major tiles, eight running sums keep eight loads in flight per thread (a narrow shard has tens of segments per
// pair and few output elements, so the pass is latency-bound), writes go through shared memory so that a warp stores
// 8-row runs of G's columns.
//
// Slab mode: xbuf != nullptr -> the sum is this device's PARTIAL result and goes to the exchange buffer
// xbuf + ((seq_base + global_iter * n_modes + mode + 1) & 1) * xcap, from where comm.cuh's exchange kernel of every
// rank collects it.
constexpr int REDUCE_ROWS = 8;
// Columns [0, C_main) come from the main instance's plan / workspace, columns [C_main, C) -- the narrow tail, if any --
// from plan_n / ws_n (tiles of M_TILE x NARROW_COLS).  C_main_override >= 0 with C_override > 0 (single-operation hook).
template <int M_TILE, int N_TILE>
__global__ void __launch_bounds__(256)
mttkrp_reduce_kernel(const MttkrpGeom g, const SchedState *__restrict__ st, const int *__restrict__ plan,
                     const double *__restrict__ ws, double *__restrict__ G, int grid_ctas, int C_override, double *xbuf,
                     unsigned long long xcap, unsigned long long seq_base, int n_modes, const int *__restrict__ plan_n,
                     const double *__restrict__ ws_n, int C_main_override) {
  pdl_enter();
  const int C = C_override > 0 ? C_override : st->C;
  const int C_main = C_override > 0 ? C_main_override : st->C_main;
  if (xbuf != nullptr) {
    const unsigned long long seq = seq_base + st->global_iter * (unsigned long long)n_modes + g.mode + 1;
    G = xbuf + (seq & 1ull) * xcap;
  }
  const int c0 = blockIdx.x * 32, m0 = blockIdx.y * REDUCE_ROWS;
  if (c0 >= C || (g.carry_fallback && st->carry_ok))
    return;
  __shared__ double t[REDUCE_ROWS][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5; // 256 threads: ty in 0..7
  {
    const int m = m0 + ty, c = c0 + tx;
    double sum = 0.0;
    if (m < g.In && c < C) {
      const bool tail = c >= C_main;
      const PlanView pv = plan_view(tail ? plan_n : plan, grid_ctas);
      const int mt = plan_tile_of(m >> 3, pv.In8, pv.m_tiles);
      const int nt = tail ? 0 : plan_tile_of(c >> 6, pv.NO, pv.n_tiles);
      const int pair = nt * pv.m_tiles + mt;
      const int s0 = pv.pair_seg0[pair], s1 = pv.pair_seg0[pair + 1];
      const size_t TE = tail ? (size_t)M_TILE * NARROW_COLS : (size_t)M_TILE * N_TILE;
      const int pitch = tail ? NARROW_COLS : N_TILE;
      const double *p = (tail ? ws_n : ws) + (size_t)s0 * TE +
                        (size_t)(m - 8 * plan_m8_start(mt, pv.In8, pv.m_tiles)) * pitch +
                        (tail ? c - C_main : c - 64 * plan_oct_start(nt, pv.NO, pv.n_tiles));
      double a[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
      int k = s0;
      for (; k + 8 <= s1; k += 8, p += 8 * TE) {
#pragma unroll
        for (int u = 0; u < 8; u++)
          a[u] += p[u * TE];
      }
      for (; k < s1; k++, p += TE) // (a static index keeps the running sums in registers)
        a[0] += *p;
      sum = ((a[0] + a[1]) + (a[2] + a[3])) + ((a[4] + a[5]) + (a[6] + a[7]));
    }
    t[ty][tx] = sum;
  }
  __syncthreads();
  { // thread -> (column = threadIdx / 8, row = threadIdx % 8)
    const int rr = threadIdx.x & (REDUCE_ROWS - 1), cc = threadIdx.x / REDUCE_ROWS;
    const int m = m0 + rr, c = c0 + cc;
    if (m < g.In && c < C)
      G[(size_t)c * g.ldG + m + g.g_row_off] = t[rr][cc];
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Cross-check kernel: one thread per output element, plain loops over the ORIGINAL tensor layout.  Not a product
// path (selected only through the CALS_B200_MTTKRP_NAIVE test hook).
struct NaiveGeom {
  int n_modes, mode;
  int dims[CALS_MAX_MODES];
  int ldF[CALS_MAX_MODES];
  long long xstride[CALS_MAX_MODES]; // element strides of the padded device copy of X
  int ldG;
  int off[CALS_MAX_MODES]; // slab mode: row offset into each factor (and into G for the output mode)
};

__global__ void mttkrp_naive_kernel(const NaiveGeom g, const SchedState *__restrict__ st, const double *__restrict__ X,
                                    const FactorPtrs fac, double *__restrict__ G, int C_override) {
  const int C = C_override > 0 ? C_override : st->C;
  const int cur = C_override > 0 ? 0 : st->cur;
  const int In = g.dims[g.mode];
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= (long long)In * C)
    return;
  const int i = (int)(tid % In), c = (int)(tid / In);
  int idx[CALS_MAX_MODES];
  for (int k = 0; k < g.n_modes; k++)
    idx[k] = 0;
  idx[g.mode] = i;
  double sum = 0.0;
  while (true) {
    long long off = 0;
    double w = 1.0;
    for (int k = 0; k < g.n_modes; k++) {
      off += idx[k] * g.xstride[k];
      if (k != g.mode)
        w *= fac.buf[cur][k][(size_t)c * g.ldF[k] + idx[k] + g.off[k]];
    }
    sum += X[off] * w;
    int k = 0;
    for (; k < g.n_modes; k++) {
      if (k == g.mode)
        continue;
      if (++idx[k] < g.dims[k])
        break;
      idx[k] = 0;
    }
    if (k == g.n_modes)
      break;
  }
  G[(size_t)c * g.ldG + i + g.off[g.mode]] = sum;
}

} // namespace calsb200
