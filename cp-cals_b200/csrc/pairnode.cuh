// Pair nodes: a one-level dimension tree over the modes.  Two modes take their MTTKRPs from ONE tensor-sized
// contraction T that does not involve either of their factors:
//
//   3 modes (pair = modes 1, 2):   T[(i1,i2), c] = sum_{i0} X[i0,i1,i2] * A_0[i0,c]           pair_gemm_kernel (FP64 tensor cores)
//   4 modes (pairs (0,1), (2,3)):  T0[(i0,i1), c] = sum_{i2,i3} X * A_2[i2,c] * A_3[i3,c]      mttkrp_dmma_kernel on a 3-way view
//                                  T1[(i2,i3), c] = sum_{i0,i1} X * A_0[i0,c] * A_1[i1,c]      (set up in engine.cu)
//   leaves, for a pair (f, s) with T rows (i_f, i_s), i_f fastest:
//                                  G_f[i_f, c] = sum_{i_s} T[(i_f,i_s), c] * A_s[i_s, c]        pair_leaf_slow_kernel (HBM-bound)
//                                  G_s[i_s, c] = sum_{i_f} T[(i_f,i_s), c] * A_f[i_f, c]        pair_leaf_fast_kernel (HBM-bound)
//   3 modes: the first leaf rides in the epilogue of pair_gemm_kernel (A_s is not touched between the contraction and
//   the leaf): a tile of T covers 8 values of i_f x WM values of i_s, every thread multiplies its accumulators by A_s
//   and sums them over the tile's i_s, and pair_partial_reduce_kernel adds the ceil(E2 / WM) partial results per
//   element in fixed order -- T is then read once per iteration instead of twice.
//
// ALS updates mode f, then mode s, and T holds neither factor, so both leaves see exactly the factors the reference's
// per-mode MTTKRPs see (src/cals.cpp:214-222 calls mttkrp::mttkrp once per mode): the sums are the same, only their
// association differs.  An ALS iteration then costs two tensor-sized contractions instead of three (four).  This is the
// reference's own two-step idea (mttkrp_twostep0/1, src/utils/mttkrp.cpp:460-553: "mode1/TS0 uses the same T as mode0/TS0")
// carried across modes; T lives in HBM.  CalsParams::mttkrp_method == MTTKRP selects one full MTTKRP per mode instead.
//
// Multi-sweep dimension tree (3 modes, engine.cu: run_loop; Ma & Solomonik, IPDPS 2021): the same kernels contract any
// mode c -- T = X x_c A_c, rows (i_{c+1}, i_{c+2}), first leaf to mode c+1, second leaf to mode c+2 (indices mod 3) --
// from a 3-D view of the tensor with mode c contiguous (PairGeom / PairMaps carry the roles).  Even passes contract
// modes 2 and 1, odd passes mode 0; the second leaf of the mode-1 contraction updates mode 0 in the NEXT pass, so two
// passes cost three contractions instead of four.
#pragma once
#include "mttkrp.cuh"

namespace calsb200 {

constexpr int PAIR_STAGES = 2;

template <int WM, int WN> struct PairCfg {
  static constexpr int M_TILE = 8 * WM;
  static constexpr int N_TILE = 8 * WN * NUM_MMA_WARPS;
  static constexpr int X_BYTES = M_TILE * KT * 8;
  static constexpr int B_BYTES = N_TILE * KT * 8;
  static constexpr int STAGE_BYTES = X_BYTES + B_BYTES;
  static constexpr int BAR_BYTES = 256;
  // fused first leaf: the tile's WM rows of the slow factor, [N_TILE][WMP]; WMP = WM rounded up to even: TMA boxes are
  // multiples of 16 bytes along the contiguous dimension and start at 16-byte granules (an odd first row makes the copy
  // fault with "illegal instruction"), so for odd WM the box starts at the even row at or below the tile's first
  static constexpr int WMP = (WM + 1) & ~1;
  static constexpr int A_BYTES = N_TILE * WMP * 8;
  static constexpr int SMEM_BYTES = PAIR_STAGES * STAGE_BYTES + BAR_BYTES + A_BYTES;
};

struct PairMaps {
  CUtensorMap X;    // 3-D view (I0, I1, I2) of the tensor in the caller's order: box [KT x 8 x WM]
  CUtensorMap B[2]; // factor of mode 0 in buffer 0 / 1: box [KT x N_TILE]
  CUtensorMap Bn[2]; // the same with a box of NARROW_COLS columns (narrow column tail, mttkrp.cuh)
  CUtensorMap A[2];  // factor of the slow mode of the pair in buffer 0 / 1: box [WMP x N_TILE] (fused first leaf)
};

struct PairGeom {
  int R;   // rows of T = I1 * I2
  int Ip;  // contracted extent (I0)
  int E1;  // extent of the fast index of a T row (I1)
  int E2;  // extent of the slow index (I2)
  int mode_fast, mode_slow; // the two modes of the pair (1 and 2)
  // Slab mode (3-mode tensor sliced along mode 1 or 2 over several GPUs): this device's T covers rows
  // [off, off + E) of the sliced mode's factor and of its G; 0 otherwise.
  int off_fast, off_slow;
  long long ldT;
  int ldF[CALS_MAX_MODES]; // leading dimensions of the factor buffers == those of G for the same mode
  // fused first leaf (3 modes, no exchange): partial results Gp[b2][c][i1], b2 = block of WM values of i2
  int fuse_slow;
  int ld_fast;         // ldF[mode_fast] (a plain field: the kernels index no parameter array at run time)
  long long gp_stride; // doubles between the partial results of consecutive b2 (= buffer columns * ldF[mode_fast])
  int carried; // second leaf from a T of the previous pass: runs only when SchedState::carry_ok (engine.cu: run_loop)
};

// T = X_(0)^T A_0.  Persistent CTAs over the (m-tile, n-tile) grid, m-tile fastest, so that the CTAs running at the
// same time share the factor tiles in L2 and the cheap tiles of the ragged last n-tile come last.  An m-tile is a patch
// of 8 values of i1 x WM values of i2 (one TMA box of the 3-D tensor view): m8 row group i of the tile is i2 = i2_0 + i,
// fragment row r is i1 = i1_0 + r.  Both operands of a K tile travel together through a two-stage TMA ring; the warp
// layout and the inner loop are those of mttkrp_dmma_kernel (mma_stage) without the outer weight.
// Epilogue: T, and -- g.fuse_slow -- the tile's share of the first leaf, Gp[b2][c][i1] = sum_i T[(i1, i2_0 + i), c] *
// A_slow[i2_0 + i, c], which a thread forms from its own accumulators (no shuffles: a thread's WM accumulators of one
// column are the WM values of i2 of one i1).
// NARROW = false: columns [0, C_main).  NARROW = true: the narrow column tail [C_main, C) (mttkrp.cuh: narrow_cols) -- one
// column tile, the eight warps split the rows of the m-tile, every warp covers the tail's n8 groups.
template <int WM, int WN, bool NARROW = false>
__global__ void __launch_bounds__(MTTKRP_THREADS, 1)
pair_gemm_kernel(const __grid_constant__ PairMaps maps, const PairGeom g, const SchedState *__restrict__ st,
                 double *__restrict__ T, double *__restrict__ Gp) {
  using Cfg = PairCfg<WM, WN>;
  constexpr int N_TILE = Cfg::N_TILE, WMP = Cfg::WMP;
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t *bars = (uint64_t *)(smem + PAIR_STAGES * Cfg::STAGE_BYTES);
  uint64_t *full = bars, *empty = bars + PAIR_STAGES;
  uint64_t *full_a = bars + 2 * PAIR_STAGES, *empty_a = full_a + 1;
  double *As = (double *)(smem + PAIR_STAGES * Cfg::STAGE_BYTES + Cfg::BAR_BYTES); // [N_TILE][WMP]
  const bool fuse = !NARROW && g.fuse_slow;

  pdl_enter();
  const int C = NARROW ? st->C : st->C_main, cur = st->cur;
  const int c_lo = NARROW ? st->C_main : 0;
  if (C - c_lo <= 0)
    return;
  const int E1b = (g.E1 + 7) >> 3, E2b = (g.E2 + WM - 1) / WM;
  const int m_tiles = E1b * E2b;
  // column tiles: the 64-column octets are split evenly over ceil(NO / 4) tiles, as in the MTTKRP plan (263 columns = 5
  // octets give tiles of 2 and 3 octets, not 4 and 1: a 1-octet tile keeps one column group per warp busy)
  const int NO = NARROW ? 1 : (C + 63) >> 6, n_tiles = (NO + OCT_TILE - 1) / OCT_TILE;
  const long long tiles = (long long)m_tiles * n_tiles;
  const int P_tiles = (g.Ip + KT - 1) / KT;
  if ((long long)blockIdx.x >= tiles)
    return;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < PAIR_STAGES; i++) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], NUM_MMA_WARPS);
    }
    mbar_init(full_a, 1);
    mbar_init(empty_a, NUM_MMA_WARPS);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp >= NUM_MMA_WARPS) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");
    if (warp != NUM_MMA_WARPS || lane != 0)
      return;
    const CUtensorMap *tmB = &maps.B[cur];
    int sidx = 0;
    uint32_t ph = 1, aph = 1;
    for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
      const int nt = (int)(t / m_tiles), mt = (int)(t - (long long)nt * m_tiles);
      const int b2 = mt / E1b, b1 = mt - b2 * E1b;
      for (int pt = 0; pt < P_tiles; pt++) {
        unsigned char *stage = smem + sidx * Cfg::STAGE_BYTES;
        mbar_wait(&empty[sidx], ph);
        if (NARROW) {
          mbar_expect_tx(&full[sidx], Cfg::X_BYTES + NARROW_COLS * KT * 8);
          tma_load_3d(stage, &maps.X, &full[sidx], pt * KT, 8 * b1, WM * b2);
          tma_load_2d(stage + Cfg::X_BYTES, &maps.Bn[cur], &full[sidx], pt * KT, c_lo);
        } else {
          mbar_expect_tx(&full[sidx], Cfg::STAGE_BYTES);
          tma_load_3d(stage, &maps.X, &full[sidx], pt * KT, 8 * b1, WM * b2);
          tma_load_2d(stage + Cfg::X_BYTES, tmB, &full[sidx], pt * KT, 64 * plan_oct_start(nt, NO, n_tiles));
        }
        if (++sidx == PAIR_STAGES) {
          sidx = 0;
          ph ^= 1;
        }
        // The slow factor's rows of this tile are needed by the epilogue only and their buffer is free once the previous
        // tile's epilogue is over: the copy is issued behind the tile's first PAIR_STAGES stage loads, which fill the ring
        // while that epilogue still runs (ahead of them, the wait would hold back the ring at every tile boundary).
        if (fuse && pt == min(PAIR_STAGES, P_tiles) - 1) {
          mbar_wait(empty_a, aph);
          aph ^= 1;
          mbar_expect_tx(full_a, Cfg::A_BYTES);
          tma_load_2d(As, &maps.A[cur], full_a, (WM * b2) & ~1, 64 * plan_oct_start(nt, NO, n_tiles));
        }
      }
    }
    return;
  }

  asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
  const int r = lane >> 2, s = lane & 3;
  double acc[WM][WN][2];
  const double ones[WN] = {1.0, 1.0, 1.0, 1.0};
  int sidx = 0;
  uint32_t ph = 0, aph = 0;
  for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
    const int nt = (int)(t / m_tiles), mt = (int)(t - (long long)nt * m_tiles);
    const int b2 = mt / E1b, b1 = mt - b2 * E1b;
    const int i1 = 8 * b1 + r, i2_0 = WM * b2; // this thread's i1; row group i of the tile is i2 = i2_0 + i
    const int c0 = 64 * plan_oct_start(nt, NO, n_tiles);
    const int nm = min(WM, g.E2 - i2_0);
    const int nn_tile = plan_nn(nt, NO, n_tiles); // octets of this tile: only their columns are this CTA's to write
    int nn = nn_tile;
    if (!NARROW && c0 + 64 * (nn - 1) + 8 * warp >= C) // this warp's n8 group of the last octet starts beyond C
      nn--;
    const int g_tail = NARROW ? min(NARROW_GROUPS, (C - c_lo + 7) >> 3) : 0;
#pragma unroll
    for (int i = 0; i < WM; i++)
#pragma unroll
      for (int j = 0; j < WN; j++)
        acc[i][j][0] = acc[i][j][1] = 0.0;
    for (int pt = 0; pt < P_tiles; pt++) {
      const double *Xs = (const double *)(smem + sidx * Cfg::STAGE_BYTES);
      const double *Bw = (const double *)(smem + sidx * Cfg::STAGE_BYTES + Cfg::X_BYTES) + warp * 8 * KT;
      const int kvalid = min(KT, g.Ip - pt * KT);
      mbar_wait(&full[sidx], ph);
      if (NARROW) {
        if (warp < nm)
          mma_narrow_stage<false>(acc[0], Xs, Bw - warp * 8 * KT, ones, (kvalid + 7) >> 3, r, s, warp, g_tail);
      } else
        mma_stage<WM, WN, false>(acc, Xs, Bw, ones, (kvalid + 7) >> 3, r, s, nm, nn);
      __syncwarp();
      if (lane == 0)
        mbar_arrive(&empty[sidx]);
      if (++sidx == PAIR_STAGES) {
        sidx = 0;
        ph ^= 1;
      }
    }
    if (NARROW) { // warp = m8 row group (= i2_0 + warp), acc[0][q] = n8 group q of the tail
      const size_t row = (size_t)i1 + (size_t)g.E1 * (i2_0 + warp);
      if (warp < nm && i1 < g.E1) {
#pragma unroll
        for (int q = 0; q < NARROW_GROUPS; q++) {
          const int col = c_lo + q * 8 + 2 * s;
          if (col < C)
            T[(size_t)col * g.ldT + row] = acc[0][q][0];
          if (col + 1 < C)
            T[(size_t)(col + 1) * g.ldT + row] = acc[0][q][1];
        }
      }
      continue; // (the narrow instance never runs together with the fused leaf: engine.cu)
    }
    // rows (i1_0 + r) + E1 * (i2_0 + i), columns c0 + 64j + 8*warp + 2s (+1): for one register the 8 lanes of equal s
    // write 8 consecutive rows of one column (64 B runs).  One pointer per column, stepped by E1 from row group to row group.
    if (fuse)
      mbar_wait(full_a, aph);
    if (i1 < g.E1) {
      double *gp = Gp + (size_t)b2 * g.gp_stride + i1;
      const int ldG = g.ld_fast;
#pragma unroll
      for (int j = 0; j < WN; j++) {
#pragma unroll
        for (int e = 0; e < 2; e++) {
          const int cl = j * 64 + warp * 8 + 2 * s + e, col = c0 + cl; // column inside the tile / of the buffer
          if (j < nn_tile && col < C) {
            double *tp = T + (size_t)col * g.ldT + ((size_t)i1 + (size_t)g.E1 * i2_0);
#pragma unroll
            for (int i = 0; i < WM; i++) {
              if (i < nm)
                *tp = acc[i][j][e];
              tp += g.E1;
            }
            if (fuse) { // accumulators of row groups beyond nm are zero, so the sum may run over all WM
              double p = 0.0;
              if (WM & 1) { // the box starts at an even row: the tile's first row is its row (WM * b2) & 1
                const double *w = As + cl * WMP + ((WM * b2) & 1);
#pragma unroll
                for (int i = 0; i < WM; i++)
                  p = fma(acc[i][j][e], w[i], p);
              } else {
                const double2 *w = reinterpret_cast<const double2 *>(As + cl * WMP);
#pragma unroll
                for (int i = 0; i < WM / 2; i++) {
                  const double2 v = w[i];
                  p = fma(acc[2 * i][j][e], v.x, p);
                  p = fma(acc[2 * i + 1][j][e], v.y, p);
                }
              }
              gp[(size_t)col * ldG] = p;
            }
          }
        }
      }
    }
    if (fuse) {
      aph ^= 1;
      __syncwarp();
      if (lane == 0)
        mbar_arrive(empty_a);
    }
  }
}

// First leaf from the partial results of pair_gemm_kernel's epilogue: G_fast[i1, c] = sum_{b2} Gp[b2][c][i1], b2 in
// ascending order (deterministic).  One thread per element, i1 fastest; the E2b partial slices are L2-resident right
// after the contraction when they fit (config 2: 25 x 3.4 MB).
__global__ void __launch_bounds__(256)
pair_partial_reduce_kernel(const PairGeom g, const SchedState *__restrict__ st, const double *__restrict__ Gp, int E2b,
                           double *__restrict__ G) {
  pdl_enter();
  const int C = st->C;
  const int c = blockIdx.y, i1 = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C || i1 >= g.E1)
    return;
  const double *p = Gp + (size_t)c * g.ld_fast + i1;
  double a[4] = {0.0, 0.0, 0.0, 0.0};
  int k = 0;
  for (; k + 4 <= E2b; k += 4, p += 4 * g.gp_stride) {
#pragma unroll
    for (int u = 0; u < 4; u++)
      a[u] += p[u * g.gp_stride];
  }
  for (; k < E2b; k++, p += g.gp_stride)
    a[0] += *p;
  G[(size_t)c * g.ld_fast + i1 + g.off_fast] = (a[0] + a[1]) + (a[2] + a[3]);
}

// Slab mode over several GPUs: a leaf's result is this device's PARTIAL sum (or its own row block) and goes to the exchange
// buffer that comm.cuh's exchange kernel collects, exactly as mttkrp_reduce_kernel does for a full MTTKRP.
struct LeafExchange {
  double *xbuf; // nullptr: write G
  unsigned long long xcap, seq_base;
  int n_modes;
};
__device__ __forceinline__ double *leaf_output(double *G, const LeafExchange &x, const SchedState *st, int mode) {
  if (x.xbuf == nullptr)
    return G;
  const unsigned long long seq = x.seq_base + st->global_iter * (unsigned long long)x.n_modes + mode + 1;
  return x.xbuf + (seq & 1ull) * x.xcap;
}

// G_fast[i1, c] = sum_{i2} T[i1 + E1*i2, c] * A_slow[i2, c].  One CTA per column and 256-row chunk of i1; thread = row.
__global__ void __launch_bounds__(256)
pair_leaf_slow_kernel(const PairGeom g, const SchedState *__restrict__ st, const FactorPtrs fac,
                      const double *__restrict__ T, double *__restrict__ G, const LeafExchange x) {
  pdl_enter();
  const int C = st->C, cur = st->cur;
  const int c = blockIdx.x;
  if (c >= C)
    return;
  G = leaf_output(G, x, st, g.mode_fast);
  extern __shared__ double wcol[]; // E2
  const double *W = fac.buf[cur][g.mode_slow] + (size_t)c * g.ldF[g.mode_slow] + g.off_slow;
  for (int k = threadIdx.x; k < g.E2; k += blockDim.x)
    wcol[k] = W[k];
  __syncthreads();
  const int i1 = blockIdx.y * blockDim.x + threadIdx.x;
  if (i1 >= g.E1)
    return;
  const double *t = T + (size_t)c * g.ldT + i1;
  double sum = 0.0;
  int k = 0;
  for (; k + 8 <= g.E2; k += 8) {
    double v[8];
#pragma unroll
    for (int u = 0; u < 8; u++)
      v[u] = __ldcs(t + (size_t)(k + u) * g.E1);
#pragma unroll
    for (int u = 0; u < 8; u++)
      sum += v[u] * wcol[k + u];
  }
  for (; k < g.E2; k++)
    sum += __ldcs(t + (size_t)k * g.E1) * wcol[k];
  G[(size_t)c * g.ldF[g.mode_fast] + i1 + g.off_fast] = sum;
}

// G_slow[i2, c] = sum_{i1} T[i1 + E1*i2, c] * A_fast[i1, c].  One CTA per column; a warp takes LEAF_ROWS values of i2 at a
// time (independent loads in flight), lanes run over i1.
constexpr int LEAF_ROWS = 4;
__global__ void __launch_bounds__(256)
pair_leaf_fast_kernel(const PairGeom g, const SchedState *__restrict__ st, const FactorPtrs fac,
                      const double *__restrict__ T, double *__restrict__ G, const LeafExchange x) {
  pdl_enter();
  const int C = st->C, cur = st->cur;
  const int c = blockIdx.x;
  if (c >= C || (g.carried && !st->carry_ok))
    return;
  G = leaf_output(G, x, st, g.mode_slow);
  extern __shared__ double wcol[]; // E1
  const double *W = fac.buf[cur][g.mode_fast] + (size_t)c * g.ldF[g.mode_fast] + g.off_fast;
  for (int k = threadIdx.x; k < g.E1; k += blockDim.x)
    wcol[k] = W[k];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const double *tc = T + (size_t)c * g.ldT;
  double *out = G + (size_t)c * g.ldF[g.mode_slow] + g.off_slow;
  for (int b2 = (blockIdx.y * nw + warp) * LEAF_ROWS; b2 < g.E2; b2 += gridDim.y * nw * LEAF_ROWS) {
    const double *t[LEAF_ROWS];
    double sum[LEAF_ROWS];
#pragma unroll
    for (int u = 0; u < LEAF_ROWS; u++) {
      t[u] = tc + (size_t)min(b2 + u, g.E2 - 1) * g.E1; // rows beyond E2 re-read the last row; their sums are dropped
      sum[u] = 0.0;
    }
    for (int i1 = lane; i1 < g.E1; i1 += 32) {
      const double w = wcol[i1];
      double v[LEAF_ROWS];
#pragma unroll
      for (int u = 0; u < LEAF_ROWS; u++)
        v[u] = __ldcs(t[u] + i1);
#pragma unroll
      for (int u = 0; u < LEAF_ROWS; u++)
        sum[u] += v[u] * w;
    }
#pragma unroll
    for (int u = 0; u < LEAF_ROWS; u++) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1)
        sum[u] += __shfl_xor_sync(0xffffffffu, sum[u], o);
      if (lane == 0 && b2 + u < g.E2)
        out[b2 + u] = sum[u];
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Slow leaf for NARROW grids (at most LEAF_TMA_MAX_COLS columns: the per-GPU shard of a strong-scaled model set,
// BASELINE config 1): one column of T per CTA, streamed through a ring of shared-memory stages filled by 1-D TMA bulk
// copies (cp.async.bulk + mbarrier complete_tx).  With one CTA per column and a few hundred columns the whole grid is
// one wave and every CTA is a single sequential stream; the per-thread loads of pair_leaf_slow_kernel keep too few bytes
// in flight for that (measured at 255 columns of 200 x 200: 42 us, this kernel 22 us, HBM floor 13 us).  On wide grids
// the plain kernel is faster (config 2: 118 us against 167 us for the pair), as is the plain fast leaf at every width
// (measured), so those stay.
//
// A bulk copy needs 16-byte aligned source, destination and size, rows of T start at any multiple of 8 bytes (odd
// E1): a row that starts at an odd element index is copied from one element earlier and read with an offset of 1.
constexpr int LEAF_STAGES = 4;
constexpr int LEAF_TMA_MAX_COLS = 592; // 4 CTAs per SM: above this the plain kernel fills the machine by itself
constexpr int LEAF_THREADS = 256;
constexpr int LEAF_SLOW_ROWS = 8;        // rows of i2 per stage in the slow leaf
constexpr int LEAF_SLOW_PITCH = 256 + 2; // doubles per staged row slice (even, room for the alignment shift)

__device__ __forceinline__ void bulk_load_1d(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

inline size_t leaf_slow_smem(int E2) {
  return (size_t)((E2 + 1) & ~1) * 8 + (size_t)LEAF_STAGES * LEAF_SLOW_ROWS * LEAF_SLOW_PITCH * 8 + 64;
}

// G_fast[i1, c] = sum_{i2} T[i1 + E1*i2, c] * A_slow[i2, c].  grid = (columns, ceil(E1 / 256)); thread = one i1.
__global__ void __launch_bounds__(LEAF_THREADS)
pair_leaf_slow_tma_kernel(const PairGeom g, const SchedState *__restrict__ st, const FactorPtrs fac,
                      const double *__restrict__ T, double *__restrict__ G, const LeafExchange x) {
  pdl_enter();
  const int C = st->C, cur = st->cur;
  const int c = blockIdx.x;
  if (c >= C)
    return;
  G = leaf_output(G, x, st, g.mode_fast);
  extern __shared__ __align__(128) unsigned char leaf_smem[];
  const int E2p = (g.E2 + 1) & ~1;
  double *wcol = (double *)leaf_smem;                    // E2 weights
  double *ring = wcol + E2p;                             // [LEAF_STAGES][LEAF_SLOW_ROWS][LEAF_SLOW_PITCH]
  uint64_t *full = (uint64_t *)(ring + LEAF_STAGES * LEAF_SLOW_ROWS * LEAF_SLOW_PITCH);
  const int tid = threadIdx.x;
  const int i0 = blockIdx.y * 256, n_i1 = min(256, g.E1 - i0);
  const size_t col_base = (size_t)c * g.ldT + i0; // element index of (i1 = i0, i2 = 0) in T
  const int n_chunks = (g.E2 + LEAF_SLOW_ROWS - 1) / LEAF_SLOW_ROWS;
  if (tid == 0) {
    for (int q = 0; q < LEAF_STAGES; q++)
      mbar_init(&full[q], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  const double *W = fac.buf[cur][g.mode_slow] + (size_t)c * g.ldF[g.mode_slow] + g.off_slow;
  for (int k = tid; k < g.E2; k += blockDim.x)
    wcol[k] = W[k];
  __syncthreads();
  auto issue = [&](int chunk) { // thread 0: all row slices of one chunk into stage chunk % LEAF_STAGES
    const int q = chunk % LEAF_STAGES, k0 = chunk * LEAF_SLOW_ROWS, nk = min(LEAF_SLOW_ROWS, g.E2 - k0);
    uint32_t total = 0;
    for (int r = 0; r < nk; r++) {
      const size_t idx = col_base + (size_t)(k0 + r) * g.E1;
      total += (uint32_t)(((n_i1 + (int)(idx & 1)) * 8 + 15) & ~15);
    }
    mbar_expect_tx(&full[q], total);
    for (int r = 0; r < nk; r++) {
      const size_t idx = col_base + (size_t)(k0 + r) * g.E1;
      const int off = (int)(idx & 1);
      bulk_load_1d(ring + ((size_t)q * LEAF_SLOW_ROWS + r) * LEAF_SLOW_PITCH, T + (idx - off),
                   (uint32_t)(((n_i1 + off) * 8 + 15) & ~15), &full[q]);
    }
  };
  if (tid == 0)
    for (int q = 0; q < LEAF_STAGES - 1 && q < n_chunks; q++)
      issue(q);
  double sum = 0.0;
  for (int ch = 0; ch < n_chunks; ch++) {
    if (tid == 0 && ch + LEAF_STAGES - 1 < n_chunks)
      issue(ch + LEAF_STAGES - 1); // its stage was consumed in iteration ch - 1 (barrier below)
    const int q = ch % LEAF_STAGES, k0 = ch * LEAF_SLOW_ROWS, nk = min(LEAF_SLOW_ROWS, g.E2 - k0);
    mbar_wait(&full[q], (uint32_t)((ch / LEAF_STAGES) & 1));
    if (tid < n_i1) {
      const double *stg = ring + (size_t)q * LEAF_SLOW_ROWS * LEAF_SLOW_PITCH + tid;
#pragma unroll
      for (int r = 0; r < LEAF_SLOW_ROWS; r++)
        if (r < nk) {
          const int off = (int)((col_base + (size_t)(k0 + r) * g.E1) & 1);
          sum += stg[r * LEAF_SLOW_PITCH + off] * wcol[k0 + r];
        }
    }
    __syncthreads();
  }
  if (tid < n_i1)
    G[(size_t)c * g.ldF[g.mode_fast] + i0 + tid + g.off_fast] = sum;
}

} // namespace calsb200
