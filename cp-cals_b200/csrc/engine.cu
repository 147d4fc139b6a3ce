// Host side of the C ABI (include/cals_b200.h): context, device memory, tensor maps and the iteration loop that replaces
// the do/while of cals::cp_cals (reference src/cals.cpp:174-382).  No cuBLAS, no CPU fallback: every entry point fails
// with an error string when the device or the sm_100a kernels are unavailable.
#include <algorithm>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <cuda.h>
#include <cuda_runtime.h>

#include "../../include/cals_b200.h"
#include "comm.cuh"
#include "common.cuh"
#include "corcon.cuh"
#include "ls.cuh"
#include "mttkrp.cuh"
#include "pairnode.cuh"
#include "prep.cuh"
#include "sched.cuh"
#include "update.cuh"
#include "wide.cuh"

using namespace calsb200;

namespace {

std::string g_create_error;

typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct HostModel { // the factors themselves go straight into the pinned input staging (ctx::h_in) at enqueue time
  int rank, jk_mode, jk_fiber, home_col;
};

// Everything whose size depends on the number of buffer columns.
struct Buffers {
  int cols = 0;
  FactorPtrs fac{};
  double *G = nullptr;
  double *ws = nullptr;
  size_t ws_tiles = 0;
  // narrow column tail (mttkrp.cuh: narrow_cols): second, narrow instance of the contraction kernels
  bool narrow = false;
  double *ws_n = nullptr;
  MttkrpMaps maps[CALS_MAX_MODES];
  MttkrpGeom mg[CALS_MAX_MODES];
  int wm[CALS_MAX_MODES];
  PlanArgs plans{}; // per-mode work partition tables (device memory) + the inputs of mttkrp_make_plan
  // pair nodes (pairnode.cuh): two modes that take their MTTKRP from one shared contraction T.  3 modes: node k
  // contracts mode k (T from pair_gemm_kernel, rows (i_{k+1}, i_{k+2})); the one-sweep schedule uses node 0 (modes 1, 2)
  // only, the multi-sweep schedule (msdt) all three, which share one T and one Gp.  4 modes: two nodes (modes 0, 1 and
  // modes 2, 3); their T comes from mttkrp_dmma_kernel run on a 3-way view of the tensor, set up in the slots
  // n_modes + k of maps / mg / wm / plans.
  struct PairNode {
    PairGeom pg{};
    double *T = nullptr; // (E1 * E2) x cols
    double *Gp = nullptr; // fused first leaf: partial results [ceil(E2 / wm)][cols][ldF[mode_fast]]
    int slot = -1;       // -1: pair_gemm_kernel
    PairMaps maps;       // pair_gemm_kernel only
    int wm = 0;          // its tile height
  };
  bool tree = false;
  bool msdt = false;
  int n_nodes = 0;
  PairNode node[3];
  int node_of[CALS_MAX_MODES] = {}; // one-sweep schedule: node that serves mode n, -1: the mode runs its own MTTKRP
  std::vector<void *> allocs;
};

} // namespace

struct cals_b200_ctx {
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  PFN_encodeTiled encode = nullptr;

  // tensor.  geo.dims are the extents of the FACTORS (the whole problem); xd are the extents of the tensor held by this
  // device: equal to geo.dims, except for the sliced mode in slab mode, where the device holds rows
  // [roff, roff + xd) of that mode (BASELINE config 5).
  Geom geo{};
  int xd[CALS_MAX_MODES] = {};
  int roff[CALS_MAX_MODES] = {};
  int slice_mode = -1;
  long long nX = 0;
  double *Xp = nullptr; // original order, pitch ldX0
  double *Xt = nullptr; // modes 0 and 1 swapped, pitch ldX1
  double *Xq = nullptr; // 4 modes, whole tensor on this device: mode pairs (0,1) and (2,3) exchanged, pitch ldXq
  double *Xr = nullptr; // 3 modes, multi-sweep schedule: mode order (2, 0, 1), pitch ldXr (made by the first run using it)
  int ldX0 = 0, ldX1 = 0, ldXq = 0, ldXr = 0;
  double *jk_norms = nullptr; // dims[0]
  double *d_norm = nullptr;
  double x_norm = 0.0;        // host copy of ||X||; valid only when x_norm_valid
  bool x_norm_valid = false;  // false between an (asynchronous) set_tensor and the first synchronising call
  bool x_norm_override = false; // cals_b200_set_tensor_norm: the host value wins over the device-computed one
  double *h_norm = nullptr;   // pinned landing place of the device-computed norm
  bool have_tensor = false;

  // params
  int buffer_cols = 4200;
  int max_iter = 200;
  double tol = 1e-7;
  unsigned flags = 0;
  int timing = 0;
  int variant = CALS_B200_MTTKRP_DMMA;
  int pair_node = 1; // cals_b200_set_pair_node
  bool pdl = false;  // programmatic dependent launch for the kernels of the iteration chain (set per run)

  // models
  std::vector<HostModel> hmodels;
  std::vector<ModelDesc> hdesc;
  int total_cols = 0, max_rank = 0;
  // models above the shared-memory update kernel's rank bound (wide.cuh); narrow_rank: largest rank at or below it
  int narrow_rank = 0, n_wide = 0, wide_min_rank = 0, wide_max_rank = 0;
  long long gram_doubles = 0;
  bool uploaded = false;
  bool results_fresh = false;
  bool fitted = false; // the home matrices and d_lambda hold the fitted models of the current queue (run / rerun)

  // run-time device state
  Buffers bufs;
  double *home0[CALS_MAX_MODES] = {}; // pristine copy of the initial home matrices (for rerun)
  ModelDesc *d_models = nullptr;
  SchedState *d_st = nullptr;
  int *d_live = nullptr, *d_live_tmp = nullptr, *d_gather = nullptr, *d_evict = nullptr;
  double *d_gram = nullptr, *d_lambda = nullptr;
  long long *d_update_prof = nullptr; // CALS_B200_UPDATE_PROF (never freed: tuning aid)
  // line search (CalsParams::line_search*, reference include/cals.h:153-156)
  int ls_enabled = 0, ls_method = 0, ls_interval = 5;
  double ls_step = 0.0;
  double *ls_prev[CALS_MAX_MODES] = {}, *ls_backup[CALS_MAX_MODES] = {};
  double *ls_prev_lambda = nullptr, *ls_backup_lambda = nullptr, *ls_partial = nullptr;
  unsigned long long last_ls_performed = 0, last_ls_failed = 0;
  unsigned char *d_active = nullptr;       // NNLS active sets of all queued models (ModelDesc::act_off)
  std::vector<unsigned char> h_active;     // host image: all 1 unless set through cals_b200_set_model_active_set
  long long active_bytes = 0;
  int *h_flags = nullptr, *d_flags = nullptr;
  unsigned *d_iter_cols = nullptr; // [ITER_LOG_CAP]
  unsigned long long last_global_iter = 0;
  std::vector<void *> run_allocs;
  int run_cols = 0, run_total_cols = 0, run_models = 0;

  // pinned staging, reused from run to run: h_in = initial factors of the queued models (filled by enqueue_model, pitch
  // ldF, one column block per model in queue order), h_home = fitted factors on the way back
  double *h_in[CALS_MAX_MODES] = {};
  size_t h_in_cap[CALS_MAX_MODES] = {};
  int queued_cols = 0;
  double *h_home[CALS_MAX_MODES] = {};
  size_t h_home_cap[CALS_MAX_MODES] = {};
  double *h_lambda = nullptr;
  size_t h_lambda_cap = 0;
  ModelDesc *h_desc_pin = nullptr;
  size_t h_desc_cap = 0;
  std::vector<int> run_sig; // (dims, buffer_cols, ranks): allocations are reused while this does not change
  double *norm_partial = nullptr;
  size_t norm_partial_cap = 0;
  double *x_stage = nullptr; // dense upload target of tensors whose fastest extent is odd (padded into Xp by a kernel)
  size_t x_stage_cap = 0;

  // slab-mode exchange over peer memory (comm.cuh)
  int comm_rank = 0, comm_world = 1;
  void *xblock = nullptr;         // [flags | 2 x xcap doubles], one cudaMalloc so that one IPC handle covers it
  size_t xcap = 0;                // doubles per exchange buffer
  void *peer_block[CALS_MAX_PEERS] = {};
  bool peer_is_ipc[CALS_MAX_PEERS] = {};
  bool comm_connected = false;
  int cuts[CALS_MAX_PEERS + 1] = {};
  unsigned long long seq_base = 0;

  // one CALS iteration captured as a CUDA graph (the launch parameters do not change between iterations, nor between
  // runs that reuse the same allocations and options)
  // [parity of the first pass]: the multi-sweep schedule alternates two iteration bodies, every other run uses [0] only
  cudaGraphExec_t iter_graph[2] = {};
  cudaGraphExec_t batch_graph[2] = {}; // the same, several iterations per launch
  std::vector<long long> iter_graph_key;
  long long alloc_generation = 0; // bumped whenever prepare_run (re)allocates

  std::vector<cudaEvent_t> ev_pool;
  bool dmma_attr_done[16] = {};
  bool pair_attr_done[32] = {}; // [WM]: main instance, [8 + WM]: narrow instance
  // prefactor_kernel (update.cuh) runs on a forked branch: second stream, fork / join events per mode, scratch
  cudaStream_t stream2 = nullptr;
  cudaEvent_t ev_fork[CALS_MAX_MODES] = {}, ev_join[CALS_MAX_MODES] = {};
  double *d_pref = nullptr; // run allocation: max_live slots of pref_stride doubles
  // wide-model workspace (wide.cuh): wide_slots slots of wide_slot_stride doubles
  double *d_wide = nullptr;
  long long wide_slot_stride = 0;
  int wide_slots = 0, wide_ldw = 0, wide_y_rows = 0;
  bool wide_attr_done = false;
  long long pref_stride = 0;
  PrefactorParams pf[CALS_MAX_MODES];
  size_t pf_smem = 0;
  int pf_grid = 0;
  int fork_mode = -1; // mode whose prefactor branch the next launch_dmma forks between its two kernels (-1: none)

  // core consistency (corcon.cuh): the call's own workspace, kept from call to call and grown when a call needs more;
  // it never shares memory with the run
  struct CorconWs {
    double *F[CALS_MAX_MODES] = {}; // the queue's factors when no fitted models are resident
    double *P[CALS_MAX_MODES] = {};
    double *T = nullptr, *chain[2] = {};
    void *tables = nullptr;
    SchedState *st = nullptr;
    double *cc = nullptr;
    int *status = nullptr, *fail = nullptr;
    size_t cap_F[CALS_MAX_MODES] = {}, cap_P[CALS_MAX_MODES] = {}, cap_T = 0, cap_chain = 0, cap_tables = 0;
    size_t cap_st = 0, cap_models = 0;
  } cc_ws;
};

namespace {

int fail(cals_b200_ctx *c, const char *fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c)
    c->err = buf;
  else
    g_create_error = buf;
  return 1;
}

#define CU_TRY(c, expr)                                                                                               \
  do {                                                                                                                \
    cudaError_t e__ = (expr);                                                                                         \
    if (e__ != cudaSuccess)                                                                                           \
      return fail((c), "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__);                  \
  } while (0)

template <typename T> int dev_alloc(cals_b200_ctx *c, T **p, size_t n, std::vector<void *> &track) {
  void *q = nullptr;
  CU_TRY(c, cudaMalloc(&q, std::max<size_t>(n, 1) * sizeof(T)));
  track.push_back(q);
  *p = (T *)q;
  return 0;
}

template <typename T> int pinned_reserve(cals_b200_ctx *c, T **p, size_t *cap, size_t n) {
  if (*p && *cap >= n)
    return 0;
  if (*p)
    cudaFreeHost(*p);
  *p = nullptr;
  *cap = 0;
  void *q = nullptr;
  CU_TRY(c, cudaHostAlloc(&q, std::max<size_t>(n, 1) * sizeof(T), cudaHostAllocDefault));
  *p = (T *)q;
  *cap = n;
  return 0;
}

void free_all(std::vector<void *> &v) {
  for (void *p : v)
    cudaFree(p);
  v.clear();
}

// Host-side copies between the callers' matrices and the pinned staging blocks: with hundreds of models (BASELINE
// config 3: 1196 models, 37 MB each way) one thread copying column by column costs more than the PCIe transfer itself,
// so large batches are split over a few threads (contiguous ranges of models; every model's bytes are disjoint).
template <typename F> void parallel_models(size_t n_models, size_t bytes, F &&fn) {
  unsigned hw = std::thread::hardware_concurrency();
  const size_t want = std::min<size_t>({(size_t)(hw ? hw : 1), (size_t)8, bytes / ((size_t)4 << 20), n_models});
  if (want <= 1) {
    fn((size_t)0, n_models);
    return;
  }
  std::vector<std::thread> th;
  const size_t per = (n_models + want - 1) / want;
  for (size_t t = 1; t < want; t++) {
    const size_t lo = std::min(n_models, t * per), hi = std::min(n_models, (t + 1) * per);
    if (lo < hi)
      th.emplace_back([&fn, lo, hi] { fn(lo, hi); });
  }
  fn((size_t)0, std::min(n_models, per));
  for (auto &t : th)
    t.join();
}

// Launch of a kernel of the iteration chain: with c->pdl the launch carries the programmatic-stream-serialization
// attribute (common.cuh: pdl_wait / pdl_trigger), so the kernel's CTAs start while the previous kernel drains.
template <typename... KArgs, typename... Args>
cudaError_t launch_chain(cals_b200_ctx *c, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, Args &&...args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = c->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = c->pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(std::forward<Args>(args))...);
}

// The dynamic shared-memory limit that cudaFuncSetAttribute sets belongs to the kernel in this process (one per device),
// not to a context: every context launches the same kernel.  So a limit that follows the problem size (update kernel,
// TMA-fed leaf, prefactor kernel) only ever grows, to the largest size any context has asked for on that device.  A
// per-context record of the last value set let a second context with a smaller problem lower the limit below what the
// first one still launched with, and the first one's next launch failed ("invalid argument").
int raise_smem_limit(cals_b200_ctx *c, const void *kern, size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<int, const void *>, size_t> limit;
  std::lock_guard<std::mutex> lock(mu);
  size_t &cur = limit[{c->device, kern}];
  if (bytes > cur) {
    CU_TRY(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    cur = bytes;
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// tile configuration
constexpr int WN_FIXED = 4;
constexpr int LS_CHUNKS = 48; // CTAs per trial model in the explicit-error kernel

// Tallest CTA tile in m8 row groups.  6 for wide buffers (config 2, 2100 columns: 85.8 k model-iterations/s with 6,
// 84.6 k with 8).  A narrow buffer -- the per-GPU shard of a strong-scaled model set -- has n-tiles of 2 or 3 octets, whose
// stages are short against their fixed cost (barriers, weight fragments), and gains from taller tiles when the mode is
// long enough to still fill the grid: 7 measured +1.1 % on the 8-way shard of config 2 (263 columns), +1.8 % on that of
// config 4 (291), +1.4 % on the 4-way shard of config 2 (525); 100-row modes (config 1) lose 0.8 %.
// CALS_B200_WM_MAX=4..8 overrides both.
int wm_max(int In, int cols) {
  static int forced = -1;
  if (forced < 0) {
    const char *e = getenv("CALS_B200_WM_MAX");
    forced = e ? atoi(e) : 0;
    if (forced < 4 || forced > 8)
      forced = 0;
  }
  if (forced)
    return forced;
  return (cols <= 640 && In >= 200) ? 7 : 6;
}

int pick_wm(int In, int cols) {
  // m8 row groups are split evenly over ceil(In8 / tallest) m-tiles; the tile is then only as tall as that split needs,
  // so that most tiles are full and run the fully unrolled path.
  const int tallest = wm_max(In, cols);
  const int In8 = (In + 7) / 8;
  const int m_tiles = (In8 + tallest - 1) / tallest;
  const int wm = (In8 + m_tiles - 1) / m_tiles;
  return wm < 4 ? 4 : wm;
}

// Tile height of pair_gemm_kernel.  Both operands stream through the ring, so a taller tile has the better flop-per-byte
// ratio (measured at 200^3 x 2100 columns: 31.6 / 33.6 / 34.6 TFLOP/s for 40 / 48 / 64 rows); small problems want enough
// tiles to fill the last wave of the persistent grid.  Score = speed of the tile shape x fill of the waves.
int pick_pair_wm(int E1, int E2, int cols, int sms) {
  static const double shape_speed[9] = {0, 0, 0, 0, 0.88, 0.915, 0.97, 0.985, 1.0};
  const long long E1b = (E1 + 7) / 8, n_tiles = (cols + TileCfg<4, WN_FIXED>::N_TILE - 1) / TileCfg<4, WN_FIXED>::N_TILE;
  int best = 8;
  double best_score = -1.0;
  for (int wm = 8; wm >= 4; wm--) { // an m-tile is 8 values of i1 x wm values of i2
    const long long E2b = (E2 + wm - 1) / wm;
    const long long tiles = E1b * E2b * n_tiles;
    const long long waves = (tiles + sms - 1) / sms;
    const double rows_used = ((double)E1 / (double)(8 * E1b)) * ((double)E2 / (double)(E2b * wm));
    const double score = shape_speed[wm] * rows_used * (double)tiles / (double)(waves * sms);
    if (score > best_score) {
      best_score = score;
      best = wm;
    }
  }
  return best;
}

template <int WM> int smem_bytes() { return TileCfg<WM, WN_FIXED>::SMEM_BYTES; }

int tile_m(int wm) { return 8 * wm; }
constexpr int TILE_N = TileCfg<4, WN_FIXED>::N_TILE;

int encode_map(cals_b200_ctx *c, CUtensorMap *map, void *base, int rank, const cuuint64_t *dims,
               const cuuint64_t *strides_bytes, const cuuint32_t *box) {
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = c->encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, (cuuint32_t)rank, base, dims, strides_bytes, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(c, "cuTensorMapEncodeTiled failed with CUresult %d (rank %d, dims %llu %llu ..)", (int)r, rank,
                (unsigned long long)dims[0], (unsigned long long)dims[1]);
  return 0;
}

// Build per-mode geometry and TMA descriptors for a set of buffers.  Tensor extents come from c->xd (the slab held by
// this device), factor pitches from c->geo; c->roff shifts every access to the sliced mode's factor.
int build_mode_plans(cals_b200_ctx *c, Buffers &b) {
  const Geom &geo = c->geo;
  const int *xd = c->xd;
  const int N = geo.n_modes;
  for (int n = 0; n < N; n++) {
    MttkrpGeom g{};
    g.mode = n;
    g.In = xd[n];
    g.p_mode = (n == 0) ? 1 : 0;
    g.Ip = xd[g.p_mode];
    g.ldG = geo.ldF[n];
    g.g_row_off = c->roff[n];
    for (int k = 0; k < N; k++)
      g.ldF[k] = geo.ldF[k];
    int no = 0;
    long long lmul = 1, umul = 1;
    for (int k = 0; k < N; k++) {
      if (k == n || k == g.p_mode)
        continue;
      g.outer_mode[no] = k;
      g.outer_dim[no] = xd[k];
      g.outer_off[no] = c->roff[k];
      if (n != 0 && k < n) {
        g.outer_lmul[no] = (int)lmul;
        g.outer_umul[no] = 0;
        lmul *= xd[k];
      } else {
        g.outer_lmul[no] = 0;
        g.outer_umul[no] = (int)umul;
        umul *= xd[k];
      }
      no++;
    }
    g.n_outer = no;
    if (no < 1)
      return fail(c, "tensors need at least 3 modes (reference asserts the same, src/cals.cpp:52)");
    g.P_tiles = (g.Ip + KT - 1) / KT;
    g.QC = (g.outer_dim[0] + OC - 1) / OC;
    long long S = 1;
    for (int k = 1; k < no; k++)
      S *= g.outer_dim[k];
    if (S > 0x7fffffff / std::max(1, g.outer_dim[0] * g.P_tiles))
      return fail(c, "tensor too large for 32-bit chunk indices");
    g.S = (int)S;
    const int wm = pick_wm(g.In, (int)b.cols);
    b.wm[n] = wm;
    g.m_tiles = (g.In + tile_m(wm) - 1) / tile_m(wm);
    b.mg[n] = g;

    // X view (P, L', M, U)
    const long long Lp = lmul, U = umul;
    cuuint64_t dims[4], strides[3];
    cuuint32_t box[4] = {(cuuint32_t)KT, 1, (cuuint32_t)tile_m(wm), 1};
    void *base;
    if (n == 0) {
      base = c->Xt;
      dims[0] = xd[1];
      dims[1] = 1;
      dims[2] = xd[0];
      dims[3] = (cuuint64_t)U;
      strides[0] = (cuuint64_t)c->ldX1 * 8;
      strides[1] = (cuuint64_t)c->ldX1 * 8;
      strides[2] = (cuuint64_t)c->ldX1 * xd[0] * 8;
    } else {
      base = c->Xp;
      dims[0] = xd[0];
      dims[1] = (cuuint64_t)Lp;
      dims[2] = xd[n];
      dims[3] = (cuuint64_t)U;
      strides[0] = (cuuint64_t)c->ldX0 * 8;
      strides[1] = (cuuint64_t)c->ldX0 * Lp * 8;
      strides[2] = (cuuint64_t)c->ldX0 * Lp * xd[n] * 8;
    }
    if (encode_map(c, &b.maps[n].X, base, 4, dims, strides, box))
      return 1;
    for (int cu = 0; cu < 2; cu++) {
      // factor tiles: rows [roff, roff + xd) of the factor (roff is even, so the base stays 16-byte aligned)
      cuuint64_t d2[2] = {(cuuint64_t)g.Ip, (cuuint64_t)b.cols};
      cuuint64_t s2[1] = {(cuuint64_t)geo.ldF[g.p_mode] * 8};
      cuuint32_t bx[2] = {(cuuint32_t)KT, (cuuint32_t)TILE_N};
      if (encode_map(c, &b.maps[n].B[cu], b.fac.buf[cu][g.p_mode] + c->roff[g.p_mode], 2, d2, s2, bx))
        return 1;
      const int q = g.outer_mode[0];
      cuuint64_t d3[2] = {(cuuint64_t)xd[q], (cuuint64_t)b.cols};
      cuuint64_t s3[1] = {(cuuint64_t)geo.ldF[q] * 8};
      cuuint32_t bw[2] = {(cuuint32_t)OC, (cuuint32_t)TILE_N};
      if (encode_map(c, &b.maps[n].W[cu], b.fac.buf[cu][q] + c->roff[q], 2, d3, s3, bw))
        return 1;
      cuuint32_t bxn[2] = {(cuuint32_t)KT, (cuuint32_t)NARROW_COLS}, bwn[2] = {(cuuint32_t)OC, (cuuint32_t)NARROW_COLS};
      if (encode_map(c, &b.maps[n].Bn[cu], b.fac.buf[cu][g.p_mode] + c->roff[g.p_mode], 2, d2, s2, bxn) ||
          encode_map(c, &b.maps[n].Wn[cu], b.fac.buf[cu][q] + c->roff[q], 2, d3, s3, bwn))
        return 1;
    }
  }
  return 0;
}

// 4 modes: geometry and TMA descriptors of the two pair-node contractions, as slots n_modes + k of the per-mode tables.
//   slot N   (node 0, modes 0 and 1):  T0[(i0,i1), c] = sum_{i2,i3} X A_2[i2,c] A_3[i3,c]   from Xq (mode 2 contiguous)
//   slot N+1 (node 1, modes 2 and 3):  T1[(i2,i3), c] = sum_{i0,i1} X A_0[i0,c] A_1[i1,c]   from Xp (mode 0 contiguous)
// Both are the MTTKRP of the last mode of a 3-way view (P, Q, R = the node's two modes flattened) of the tensor, which is
// what mttkrp_dmma_kernel computes.
int build_node_slots(cals_b200_ctx *c, Buffers &b) {
  const Geom &geo = c->geo;
  const int N = geo.n_modes;
  for (int k = 0; k < 2; k++) {
    const int slot = N + k;
    const int p = k == 0 ? 2 : 0, q = p + 1; // contracted modes: p contiguous, q the outer one
    const int R = b.node[k].pg.R;
    const double *base = k == 0 ? c->Xq : c->Xp;
    const long long ldp = k == 0 ? c->ldXq : c->ldX0;
    MttkrpGeom g{};
    g.mode = slot;
    g.In = R;
    g.p_mode = p;
    g.Ip = c->xd[p];
    g.ldG = R;
    g.g_row_off = 0;
    for (int m = 0; m < N; m++)
      g.ldF[m] = geo.ldF[m];
    g.n_outer = 1;
    g.outer_mode[0] = q;
    g.outer_dim[0] = c->xd[q];
    g.outer_off[0] = 0;
    g.outer_lmul[0] = 1;
    g.outer_umul[0] = 0;
    g.P_tiles = (g.Ip + KT - 1) / KT;
    g.QC = (g.outer_dim[0] + OC - 1) / OC;
    g.S = 1;
    const int wm = pick_wm(R, (int)b.cols);
    b.wm[slot] = wm;
    g.m_tiles = (R + tile_m(wm) - 1) / tile_m(wm);
    b.mg[slot] = g;
    cuuint64_t dims[4] = {(cuuint64_t)c->xd[p], (cuuint64_t)c->xd[q], (cuuint64_t)R, 1};
    cuuint64_t strides[3] = {(cuuint64_t)ldp * 8, (cuuint64_t)ldp * c->xd[q] * 8, (cuuint64_t)ldp * c->xd[q] * R * 8};
    cuuint32_t box[4] = {(cuuint32_t)KT, 1, (cuuint32_t)tile_m(wm), 1};
    if (encode_map(c, &b.maps[slot].X, const_cast<double *>(base), 4, dims, strides, box))
      return 1;
    for (int cu = 0; cu < 2; cu++) {
      cuuint64_t d2[2] = {(cuuint64_t)c->xd[p], (cuuint64_t)b.cols};
      cuuint64_t s2[1] = {(cuuint64_t)geo.ldF[p] * 8};
      cuuint32_t bx[2] = {(cuuint32_t)KT, (cuuint32_t)TILE_N};
      if (encode_map(c, &b.maps[slot].B[cu], b.fac.buf[cu][p], 2, d2, s2, bx))
        return 1;
      cuuint64_t d3[2] = {(cuuint64_t)c->xd[q], (cuuint64_t)b.cols};
      cuuint64_t s3[1] = {(cuuint64_t)geo.ldF[q] * 8};
      cuuint32_t bw[2] = {(cuuint32_t)OC, (cuuint32_t)TILE_N};
      if (encode_map(c, &b.maps[slot].W[cu], b.fac.buf[cu][q], 2, d3, s3, bw))
        return 1;
      cuuint32_t bxn[2] = {(cuuint32_t)KT, (cuuint32_t)NARROW_COLS}, bwn[2] = {(cuuint32_t)OC, (cuuint32_t)NARROW_COLS};
      if (encode_map(c, &b.maps[slot].Bn[cu], b.fac.buf[cu][p], 2, d2, s2, bxn) ||
          encode_map(c, &b.maps[slot].Wn[cu], b.fac.buf[cu][q], 2, d3, s3, bwn))
        return 1;
    }
  }
  return 0;
}

// CALS_B200_FUSED_LEAF: -1 unset (the buffer shape decides), 0 / 1 forced.  Read per run -- it is part of the allocation
// signature -- so that one process can measure and test both forms of the first leaf.
int fused_leaf_knob() {
  const char *e = getenv("CALS_B200_FUSED_LEAF");
  return e ? (atoi(e) != 0 ? 1 : 0) : -1;
}

// Pair nodes need a 3- or 4-mode tensor that is whole on this device (or, 3 modes, sliced along mode 1 or 2) and factor
// columns that fit the leaf kernels' shared memory (the run loop uses them with the tensor-core MTTKRP variant only); CALS_B200_NO_PAIR_NODE=1 keeps the three per-mode MTTKRPs (A/B measurements).
bool pair_node_wanted(cals_b200_ctx *c) {
  static const bool off = getenv("CALS_B200_NO_PAIR_NODE") != nullptr;
  if (off || !c->pair_node || (c->geo.n_modes != 3 && c->geo.n_modes != 4))
    return false;
  // a sliced tensor: T of a slab is local to its GPU when the slab cuts one of the pair's own modes (3 modes: 1 or 2)
  if (c->slice_mode >= 0 && !(c->geo.n_modes == 3 && c->slice_mode >= 1))
    return false;
  for (int n = 0; n < c->geo.n_modes; n++)
    if (c->xd[n] > 5000)
      return false;
  return c->geo.n_modes == 3 || c->Xq != nullptr;
}

// CALS_B200_MSDT: -1 unset (the extents decide), 0 / 1 forced.  Read per run -- it is part of the allocation signature.
int msdt_knob() {
  const char *e = getenv("CALS_B200_MSDT");
  return e ? (atoi(e) != 0 ? 1 : 0) : -1;
}

// Shortest mode for which the multi-sweep schedule pays: the contraction over mode c writes T and its leaves read it
// back, 16 * (nX / I_c) * C bytes against 2 * nX * C flop, so a short contracted mode makes T's traffic as long as the
// contraction it saves.
constexpr int MSDT_MIN_EXTENT = 64;

// The multi-sweep schedule (run_loop) needs a 3-mode tensor whole on this device, factors that no line search rewrites
// behind the carried T, and no narrow column tail (its tiles carry no fused-leaf partials).
bool msdt_wanted(cals_b200_ctx *c) {
  static const bool narrow_instance = getenv("CALS_B200_NARROW") != nullptr;
  const int knob = msdt_knob();
  if (knob == 0 || c->geo.n_modes != 3 || c->slice_mode >= 0 || c->ls_enabled || narrow_instance)
    return false;
  return knob == 1 || std::min({c->xd[0], c->xd[1], c->xd[2]}) >= MSDT_MIN_EXTENT;
}

int build_xr(cals_b200_ctx *c) {
  const int I0 = c->xd[0], I1 = c->xd[1], I2 = c->xd[2];
  c->ldXr = round_up_int(I2, 2);
  if (!c->Xr)
    CU_TRY(c, cudaMalloc((void **)&c->Xr, (size_t)c->ldXr * I0 * I1 * 8));
  dim3 grid((unsigned)(((long long)I0 * I1 + 31) / 32), (unsigned)((I2 + 31) / 32));
  rot201_copy_kernel<<<grid, 256, 0, c->stream>>>(c->Xp, c->Xr, I0, I1, I2, c->ldX0, c->ldXr);
  CU_TRY(c, cudaGetLastError());
  return 0;
}

// 3 modes: node k contracts mode k, T[(i_f + E1 * i_s), c] = sum_{i_k} X A_k[i_k, c] with f = k+1, s = k+2 (mod 3), read
// from a 3-D view (i_k, i_f, i_s) of the tensor with mode k contiguous: Xp for k = 0, Xt (storage order i1, i0, i2) with
// its two outer strides swapped for k = 1, Xr for k = 2.
int build_pair_node3(cals_b200_ctx *c, Buffers &b, int k, int cols) {
  const Geom &geo = c->geo;
  Buffers::PairNode &nd = b.node[k];
  const int mf = (k + 1) % 3, ms = (k + 2) % 3;
  PairGeom &pg = nd.pg;
  pg = PairGeom{};
  pg.E1 = c->xd[mf];
  pg.E2 = c->xd[ms];
  pg.R = pg.E1 * pg.E2;
  pg.ldT = pg.R;
  pg.Ip = c->xd[k];
  pg.mode_fast = mf;
  pg.mode_slow = ms;
  pg.off_fast = c->roff[mf];
  pg.off_slow = c->roff[ms];
  for (int m = 0; m < 3; m++)
    pg.ldF[m] = geo.ldF[m];
  nd.slot = -1;
  nd.wm = pick_pair_wm(pg.E1, pg.E2, cols, c->sm_count);
  // m-tile = 8 values of i_f x wm values of i_s (pairnode.cuh): one box of the 3-D view
  const cuuint64_t I0 = c->xd[0], I1 = c->xd[1];
  cuuint64_t dx[3] = {(cuuint64_t)pg.Ip, (cuuint64_t)pg.E1, (cuuint64_t)pg.E2}, sx[2];
  double *base;
  if (k == 0) {
    base = c->Xp;
    sx[0] = (cuuint64_t)c->ldX0 * 8;
    sx[1] = (cuuint64_t)c->ldX0 * I1 * 8;
  } else if (k == 1) {
    base = c->Xt;
    sx[0] = (cuuint64_t)c->ldX1 * I0 * 8;
    sx[1] = (cuuint64_t)c->ldX1 * 8;
  } else {
    base = c->Xr;
    sx[0] = (cuuint64_t)c->ldXr * 8;
    sx[1] = (cuuint64_t)c->ldXr * I0 * 8;
  }
  cuuint32_t bx[3] = {(cuuint32_t)KT, 8, (cuuint32_t)nd.wm};
  if (encode_map(c, &nd.maps.X, base, 3, dx, sx, bx))
    return 1;
  // The first leaf rides in the contraction's epilogue (pairnode.cuh) unless its result is a partial sum that goes
  // to the exchange buffer (sliced tensor over several GPUs).  Measured (fused against separate
  // pass): config 2 86.5 k against 84.8 k model-iterations/s, config 1 365 k against 341 k; the 8-way shard of
  // config 2 -- 263 columns, where the TMA-fed slow leaf already streams T at HBM speed and the epilogue is a larger
  // share of the short tiles -- 57.6 k against 58.0 k, so a narrow buffer over a large T keeps the separate pass.
  // CALS_B200_FUSED_LEAF=0 / 1 forces either.
  const int fl = fused_leaf_knob();
  static const bool narrow_instance = getenv("CALS_B200_NARROW") != nullptr; // (its tiles carry no partials)
  const bool narrow_big = cols <= LEAF_TMA_MAX_COLS && (size_t)pg.R * cols * 8 > ((size_t)32 << 20);
  const bool want_fused = fl >= 0 ? fl != 0 : !narrow_big;
  pg.fuse_slow = (want_fused && !narrow_instance && !(c->slice_mode >= 0 && c->comm_world > 1)) ? 1 : 0;
  pg.ld_fast = geo.ldF[mf];
  pg.gp_stride = (long long)cols * geo.ldF[mf];
  for (int cu = 0; cu < 2; cu++) {
    if (pg.fuse_slow) { // the slow factor's rows of a tile: [wm rounded up to even] x TILE_N
      cuuint64_t da[2] = {(cuuint64_t)pg.E2, (cuuint64_t)cols};
      cuuint64_t sa[1] = {(cuuint64_t)geo.ldF[ms] * 8};
      cuuint32_t ba[2] = {(cuuint32_t)((nd.wm + 1) & ~1), (cuuint32_t)TILE_N};
      if (encode_map(c, &nd.maps.A[cu], b.fac.buf[cu][ms] + pg.off_slow, 2, da, sa, ba))
        return 1;
    }
    cuuint64_t d2[2] = {(cuuint64_t)pg.Ip, (cuuint64_t)cols};
    cuuint64_t s2[1] = {(cuuint64_t)geo.ldF[k] * 8};
    cuuint32_t b2[2] = {(cuuint32_t)KT, (cuuint32_t)TILE_N}, b2n[2] = {(cuuint32_t)KT, (cuuint32_t)NARROW_COLS};
    if (encode_map(c, &nd.maps.B[cu], b.fac.buf[cu][k] + c->roff[k], 2, d2, s2, b2) ||
        encode_map(c, &nd.maps.Bn[cu], b.fac.buf[cu][k] + c->roff[k], 2, d2, s2, b2n))
      return 1;
  }
  return 0;
}

int alloc_buffers(cals_b200_ctx *c, Buffers &b, int cols, bool with_home_cols, int home_cols) {
  const Geom &geo = c->geo;
  b.cols = cols;
  int max_ld = 0;
  for (int n = 0; n < geo.n_modes; n++) {
    max_ld = std::max(max_ld, geo.ldF[n]);
    for (int cu = 0; cu < 2; cu++) {
      if (dev_alloc(c, &b.fac.buf[cu][n], (size_t)geo.ldF[n] * cols, b.allocs))
        return 1;
      CU_TRY(c, cudaMemsetAsync(b.fac.buf[cu][n], 0, (size_t)geo.ldF[n] * cols * 8, c->stream));
    }
    if (with_home_cols) {
      if (dev_alloc(c, &b.fac.home[n], (size_t)geo.ldF[n] * home_cols, b.allocs))
        return 1;
      CU_TRY(c, cudaMemsetAsync(b.fac.home[n], 0, (size_t)geo.ldF[n] * home_cols * 8, c->stream));
    }
  }
  if (dev_alloc(c, &b.G, (size_t)max_ld * cols, b.allocs))
    return 1;
  if (build_mode_plans(c, b))
    return 1;

  // pair nodes (run buffers only; the single-MTTKRP test hook stays per mode)
  const int N = geo.n_modes;
  b.tree = false;
  b.msdt = false;
  b.n_nodes = 0;
  for (int n = 0; n < CALS_MAX_MODES; n++)
    b.node_of[n] = -1;
  if (with_home_cols && pair_node_wanted(c)) {
    size_t free_b = 0, total_b = 0;
    CU_TRY(c, cudaMemGetInfo(&free_b, &total_b));
    auto fits = [&](size_t need) { // T plus, for 4 modes, a partial-tile workspace of similar size
      return 2 * need + ((size_t)2 << 30) < free_b;
    };
    if (N == 3) {
      // one-sweep schedule: node 0 = modes (1,2).  Multi-sweep: nodes 0, 1, 2 with one T and one Gp of the largest size,
      // and the (2, 0, 1) copy of the tensor.
      const size_t R0 = (size_t)c->xd[1] * c->xd[2];
      const size_t R_max = std::max({R0, (size_t)c->xd[2] * c->xd[0], (size_t)c->xd[0] * c->xd[1]});
      const size_t xr_bytes = c->Xr ? 0 : (size_t)round_up_int(c->xd[2], 2) * c->xd[0] * c->xd[1] * 8;
      b.msdt = msdt_wanted(c) && fits(R_max * cols * 8 + xr_bytes);
      if (b.msdt || fits(R0 * cols * 8)) {
        if (b.msdt && !c->Xr && build_xr(c))
          return 1;
        b.n_nodes = b.msdt ? 3 : 1;
        double *T = nullptr;
        // + 2: the leaf kernels' bulk copies read 16-byte granules and may touch one double past the last row
        if (dev_alloc(c, &T, (b.msdt ? R_max : R0) * cols + 2, b.allocs))
          return 1;
        size_t gp = 0;
        for (int k = 0; k < b.n_nodes; k++) {
          if (build_pair_node3(c, b, k, cols))
            return 1;
          const PairGeom &pg = b.node[k].pg;
          b.node[k].T = T;
          if (pg.fuse_slow)
            gp = std::max(gp, (size_t)(pg.E2 + b.node[k].wm - 1) / b.node[k].wm * (size_t)pg.gp_stride);
        }
        double *Gp = nullptr;
        if (gp > 0 && dev_alloc(c, &Gp, gp, b.allocs))
          return 1;
        for (int k = 0; k < b.n_nodes; k++)
          b.node[k].Gp = Gp;
        b.node_of[1] = b.node_of[2] = 0;
        b.tree = true;
      }
    } else if (fits(((size_t)c->xd[0] * c->xd[1] + (size_t)c->xd[2] * c->xd[3]) * cols * 8)) {
      // 4 modes: node 0 = modes (0,1), node 1 = modes (2,3)
      b.n_nodes = 2;
      for (int k = 0; k < b.n_nodes; k++) {
        Buffers::PairNode &nd = b.node[k];
        const int mf = 2 * k;
        nd.pg = PairGeom{};
        nd.pg.E1 = c->xd[mf];
        nd.pg.E2 = c->xd[mf + 1];
        nd.pg.R = c->xd[mf] * c->xd[mf + 1];
        nd.pg.ldT = nd.pg.R;
        nd.pg.mode_fast = mf;
        nd.pg.mode_slow = mf + 1;
        nd.pg.off_fast = c->roff[mf];
        nd.pg.off_slow = c->roff[mf + 1];
        for (int m = 0; m < N; m++)
          nd.pg.ldF[m] = geo.ldF[m];
        nd.slot = N + k;
        // + 2: the leaf kernels' bulk copies read 16-byte granules and may touch one double past the last row
        if (dev_alloc(c, &nd.T, (size_t)nd.pg.R * cols + 2, b.allocs))
          return 1;
        b.node_of[mf] = b.node_of[mf + 1] = k;
      }
      b.tree = true;
      if (build_node_slots(c, b))
        return 1;
    }
    for (int k = 0; k < b.n_nodes; k++) // dynamic shared memory of the TMA-fed leaf kernel (ring of stages)
      if (raise_smem_limit(c, (const void *)pair_leaf_slow_tma_kernel, leaf_slow_smem(b.node[k].pg.E2)))
        return 1;
  }

  size_t tiles = 0, tile_elems = 0;
  const int n_tiles_max = ((cols + 63) / 64 + OCT_TILE - 1) / OCT_TILE;
  const int n_plans = N + ((b.tree && N == 4) ? 2 : 0);
  b.plans = PlanArgs{};
  b.plans.n_modes = n_plans;
  b.plans.G = c->sm_count;
  if (dev_alloc(c, &b.plans.built_for, (size_t)2 * CALS_MAX_MODES, b.allocs))
    return 1;
  CU_TRY(c, cudaMemsetAsync(b.plans.built_for, 0xff, 2 * CALS_MAX_MODES * sizeof(int), c->stream));
  // Narrow column tail (mttkrp.cuh: narrow_cols): a second, row-splitting instance of the contraction kernels for a
  // tail of at most 32 columns.  OFF unless CALS_B200_NARROW=1: measured on the B200 the extra persistent kernel --
  // it streams X once more, and its stages are all barrier and TMA overhead -- costs as much as the slot it saves in
  // the main instance (8-way shard of config 2, 263 columns: 56.6 k -> 54.9 k model-iterations/s; config 1, 220 columns:
  // 339 k -> 305 k; 8-way shard of config 3: 253 k -> 239 k).  The main instances are bit-for-bit the same code either way.
  static const bool narrow_wanted = getenv("CALS_B200_NARROW") != nullptr;
  b.narrow = narrow_wanted && narrow_cols(cols) > 0;
  for (int n = 0; n < n_plans; n++) {
    const int pairs_max = b.mg[n].m_tiles * n_tiles_max;
    tiles = std::max(tiles, (size_t)(c->sm_count + pairs_max + 2));
    tile_elems = std::max(tile_elems, (size_t)tile_m(b.wm[n]) * TILE_N);
    if (dev_alloc(c, &b.plans.plan[n], (size_t)plan_capacity(c->sm_count, pairs_max), b.allocs))
      return 1;
    if (b.narrow && dev_alloc(c, &b.plans.plan_narrow[n], (size_t)plan_capacity(c->sm_count, b.mg[n].m_tiles), b.allocs))
      return 1;
    b.plans.shape[n].In = b.mg[n].In;
    b.plans.shape[n].WM = b.wm[n];
    b.plans.shape[n].Ip = b.mg[n].Ip;
    b.plans.shape[n].Iq = b.mg[n].outer_dim[0];
    b.plans.shape[n].S = b.mg[n].S;
    const long long tp = (long long)b.mg[n].P_tiles * b.mg[n].S * b.mg[n].outer_dim[0];
    if (tp * pairs_max > 0x7fffffffLL)
      return fail(c, "tensor too large for 32-bit chunk indices");
    if (tp != plan_tp(b.plans.shape[n]))
      return fail(c, "internal error: chunk count mismatch");
  }
  b.ws_tiles = tiles;
  if (dev_alloc(c, &b.ws, tiles * tile_elems, b.allocs))
    return 1;
  if (b.narrow) { // partial tiles of the narrow instance: M_TILE x NARROW_COLS, at most one per CTA and one per m-tile
    size_t mt_max = 0;
    for (int n = 0; n < n_plans; n++)
      mt_max = std::max(mt_max, (size_t)b.mg[n].m_tiles);
    if (dev_alloc(c, &b.ws_n, (size_t)(c->sm_count + mt_max + 2) * 64 * NARROW_COLS, b.allocs))
      return 1;
  }
  return 0;
}

template <int WM> int launch_pair_gemm_wm(cals_b200_ctx *c, Buffers &b, const Buffers::PairNode &nd, bool attr_only) {
  auto kern = pair_gemm_kernel<WM, WN_FIXED>;
  constexpr int smem = PairCfg<WM, WN_FIXED>::SMEM_BYTES;
  if (!c->pair_attr_done[WM]) {
    CU_TRY(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    c->pair_attr_done[WM] = true;
  }
  auto kern_n = pair_gemm_kernel<WM, WN_FIXED, true>;
  if (b.narrow && !c->pair_attr_done[8 + WM]) {
    CU_TRY(c, cudaFuncSetAttribute(kern_n, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    c->pair_attr_done[8 + WM] = true;
  }
  if (!attr_only) {
    CU_TRY(c, launch_chain(c, kern, dim3(c->sm_count), dim3(MTTKRP_THREADS), (size_t)smem, nd.maps, nd.pg,
                           (const SchedState *)c->d_st, nd.T, nd.Gp));
    if (b.narrow)
      CU_TRY(c, launch_chain(c, kern_n, dim3(c->sm_count), dim3(MTTKRP_THREADS), (size_t)smem, nd.maps, nd.pg,
                             (const SchedState *)c->d_st, nd.T, nd.Gp));
  }
  return 0;
}

// T of 3-mode node k: the tensor contracted over mode k (attr_only: just make sure the kernel's shared-memory attribute
// is set, outside of a graph capture)
int launch_pair_gemm(cals_b200_ctx *c, Buffers &b, int k, bool attr_only = false) {
  const Buffers::PairNode &nd = b.node[k];
  switch (nd.wm) {
  case 4:
    return launch_pair_gemm_wm<4>(c, b, nd, attr_only);
  case 5:
    return launch_pair_gemm_wm<5>(c, b, nd, attr_only);
  case 6:
    return launch_pair_gemm_wm<6>(c, b, nd, attr_only);
  case 7:
    return launch_pair_gemm_wm<7>(c, b, nd, attr_only);
  default:
    return launch_pair_gemm_wm<8>(c, b, nd, attr_only);
  }
}

double *exchange_data(cals_b200_ctx *c);

// MTTKRP of mode n (one of the two modes of node k) from the node's T.  carried: the second leaf of a T made in the
// previous pass, which runs only when the scheduler found that T still valid (SchedState::carry_ok).
int launch_pair_leaf(cals_b200_ctx *c, Buffers &b, int k, int n, bool exchange, bool carried = false) {
  const Buffers::PairNode &nd = b.node[k];
  PairGeom pg = nd.pg;
  pg.carried = carried ? 1 : 0;
  LeafExchange x{};
  x.xbuf = exchange ? exchange_data(c) : nullptr;
  x.xcap = (unsigned long long)c->xcap;
  x.seq_base = c->seq_base;
  x.n_modes = c->geo.n_modes;
  if (n == pg.mode_fast && pg.fuse_slow && nd.slot < 0 && !exchange) {
    // the contraction's epilogue has left ceil(E2 / wm) partial results per element
    dim3 grid((unsigned)((pg.E1 + 255) / 256), (unsigned)b.cols);
    CU_TRY(c, launch_chain(c, pair_partial_reduce_kernel, grid, dim3(256), (size_t)0, pg, (const SchedState *)c->d_st,
                           (const double *)nd.Gp, (pg.E2 + nd.wm - 1) / nd.wm, b.G));
  } else if (n == pg.mode_fast) {
    dim3 grid((unsigned)b.cols, (unsigned)((pg.E1 + 255) / 256));
    if (b.cols <= LEAF_TMA_MAX_COLS) // narrow grid: one TMA-fed stream per column
      CU_TRY(c, launch_chain(c, pair_leaf_slow_tma_kernel, grid, dim3(LEAF_THREADS), leaf_slow_smem(pg.E2), pg,
                             (const SchedState *)c->d_st, b.fac, (const double *)nd.T, b.G, x));
    else
      CU_TRY(c, launch_chain(c, pair_leaf_slow_kernel, grid, dim3(256), (size_t)pg.E2 * 8, pg,
                             (const SchedState *)c->d_st, b.fac, (const double *)nd.T, b.G, x));
  } else {
    dim3 grid((unsigned)b.cols, 1);
    CU_TRY(c, launch_chain(c, pair_leaf_fast_kernel, grid, dim3(256), (size_t)pg.E1 * 8, pg, (const SchedState *)c->d_st,
                           b.fac, (const double *)nd.T, b.G, x));
  }
  return 0;
}

double *exchange_data(cals_b200_ctx *c) { return (double *)((char *)c->xblock + COMM_FLAG_BYTES); }

template <int WM> int set_dmma_attr(cals_b200_ctx *c) {
  if (!c->dmma_attr_done[WM]) {
    CU_TRY(c, cudaFuncSetAttribute(mttkrp_dmma_kernel<WM, WN_FIXED, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   smem_bytes<WM>()));
    CU_TRY(c, cudaFuncSetAttribute(mttkrp_dmma_kernel<WM, WN_FIXED, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   smem_bytes<WM>()));
    c->dmma_attr_done[WM] = true;
  }
  return 0;
}

int ensure_dmma_attr(cals_b200_ctx *c, int wm) {
  switch (wm) {
  case 4:
    return set_dmma_attr<4>(c);
  case 5:
    return set_dmma_attr<5>(c);
  case 6:
    return set_dmma_attr<6>(c);
  case 7:
    return set_dmma_attr<7>(c);
  default:
    return set_dmma_attr<8>(c);
  }
}

// Fork: prefactor_kernel of mode n on the second stream, ordered after everything enqueued on the main stream so far;
// join_prefactor makes the main stream wait for it (in a stream capture both become graph edges).
int fork_prefactor(cals_b200_ctx *c, int n) {
  CU_TRY(c, cudaEventRecord(c->ev_fork[n], c->stream));
  CU_TRY(c, cudaStreamWaitEvent(c->stream2, c->ev_fork[n], 0));
  prefactor_kernel<<<c->pf_grid, PREFACTOR_THREADS, c->pf_smem, c->stream2>>>(c->pf[n]);
  CU_TRY(c, cudaEventRecord(c->ev_join[n], c->stream2));
  return 0;
}
int join_prefactor(cals_b200_ctx *c, int n) {
  CU_TRY(c, cudaStreamWaitEvent(c->stream, c->ev_join[n], 0));
  return 0;
}

template <int WM>
int launch_dmma(cals_b200_ctx *c, Buffers &b, int n, int C_override, bool exchange, bool skip_reduce, double *out,
                bool carry_fallback) {
  MttkrpGeom mg = b.mg[n];
  mg.carry_fallback = carry_fallback ? 1 : 0;
  auto kern = mttkrp_dmma_kernel<WM, WN_FIXED, false>;
  auto kern_n = mttkrp_dmma_kernel<WM, WN_FIXED, true>;
  if (set_dmma_attr<WM>(c))
    return 1;
  const int G = c->sm_count;
  // single-operation hook (C_override > 0): the split of the columns is made here; iteration path: by the scheduler
  const int tail = (C_override > 0 && b.narrow) ? narrow_cols(C_override) : 0;
  const int C_main_ov = C_override > 0 ? C_override - tail : 0;
  if (C_override <= 0 || C_main_ov > 0)
    CU_TRY(c, launch_chain(c, kern, dim3(G), dim3(MTTKRP_THREADS), (size_t)smem_bytes<WM>(), b.maps[n], mg,
                           (const SchedState *)c->d_st, b.fac, (const int *)b.plans.plan[n], b.ws, C_main_ov, 0));
  if (b.narrow && (C_override <= 0 || tail > 0))
    CU_TRY(c, launch_chain(c, kern_n, dim3(G), dim3(MTTKRP_THREADS), (size_t)smem_bytes<WM>(), b.maps[n], mg,
                           (const SchedState *)c->d_st, b.fac, (const int *)b.plans.plan_narrow[n], b.ws_n, C_override,
                           C_main_ov));
  if (skip_reduce) // the update kernel sums the partial tiles itself
    return 0;
  if (c->fork_mode >= 0) { // the prefactor branch runs next to the reduce pass, not next to the persistent DMMA kernel
    const int fm = c->fork_mode;
    c->fork_mode = -1;
    if (fork_prefactor(c, fm))
      return 1;
  }
  const int cols = C_override > 0 ? C_override : b.cols;
  dim3 rg((cols + 31) / 32, (b.mg[n].In + REDUCE_ROWS - 1) / REDUCE_ROWS);
  CU_TRY(c, launch_chain(c, mttkrp_reduce_kernel<8 * WM, TILE_N>, rg, dim3(256), (size_t)0, mg,
                         (const SchedState *)c->d_st, (const int *)b.plans.plan[n], (const double *)b.ws, out, G,
                         C_override, exchange ? exchange_data(c) : (double *)nullptr, (unsigned long long)c->xcap,
                         (unsigned long long)c->seq_base, c->geo.n_modes, (const int *)b.plans.plan_narrow[n],
                         (const double *)b.ws_n, C_main_ov));
  return 0;
}

// n < n_modes: MTTKRP of mode n into G.  n >= n_modes: contraction of a pair node's slot into `out` (its T).
// carry_fallback: the kernels run only when the carried T is not valid (SchedState::carry_ok == 0).
int launch_mttkrp(cals_b200_ctx *c, Buffers &b, int n, int C_override, int variant, bool exchange = false,
                  bool skip_reduce = false, double *out = nullptr, bool carry_fallback = false) {
  if (!out)
    out = b.G;
  if (variant == CALS_B200_MTTKRP_NAIVE) {
    if (exchange)
      return fail(c, "the naive MTTKRP variant does not support a sliced tensor over several GPUs");
    NaiveGeom ng{};
    ng.n_modes = c->geo.n_modes;
    ng.mode = n;
    long long stride = 1;
    for (int k = 0; k < ng.n_modes; k++) {
      ng.dims[k] = c->xd[k];
      ng.ldF[k] = c->geo.ldF[k];
      ng.off[k] = c->roff[k];
      ng.xstride[k] = stride;
      stride *= (k == 0) ? c->ldX0 : c->xd[k];
    }
    ng.ldG = c->geo.ldF[n];
    const int cols = C_override > 0 ? C_override : b.cols;
    const long long total = (long long)ng.dims[n] * cols;
    mttkrp_naive_kernel<<<(unsigned)((total + 127) / 128), 128, 0, c->stream>>>(ng, c->d_st, c->Xp, b.fac, b.G,
                                                                                 C_override);
    return 0;
  }
  switch (b.wm[n]) {
  case 4:
    return launch_dmma<4>(c, b, n, C_override, exchange, skip_reduce, out, carry_fallback);
  case 5:
    return launch_dmma<5>(c, b, n, C_override, exchange, skip_reduce, out, carry_fallback);
  case 6:
    return launch_dmma<6>(c, b, n, C_override, exchange, skip_reduce, out, carry_fallback);
  case 7:
    return launch_dmma<7>(c, b, n, C_override, exchange, skip_reduce, out, carry_fallback);
  default:
    return launch_dmma<8>(c, b, n, C_override, exchange, skip_reduce, out, carry_fallback);
  }
}

int ensure_dummy_state(cals_b200_ctx *c) {
  if (!c->d_st) {
    CU_TRY(c, cudaMalloc((void **)&c->d_st, sizeof(SchedState)));
    CU_TRY(c, cudaMemset(c->d_st, 0, sizeof(SchedState)));
  }
  if (!c->d_iter_cols)
    CU_TRY(c, cudaMalloc((void **)&c->d_iter_cols, (size_t)ITER_LOG_CAP * sizeof(unsigned)));
  return 0;
}

void drop_iteration_graph(cals_b200_ctx *c) {
  for (int p = 0; p < 2; p++) {
    if (c->iter_graph[p])
      cudaGraphExecDestroy(c->iter_graph[p]);
    if (c->batch_graph[p])
      cudaGraphExecDestroy(c->batch_graph[p]);
    c->iter_graph[p] = nullptr;
    c->batch_graph[p] = nullptr;
  }
  c->iter_graph_key.clear();
}

void release_run(cals_b200_ctx *c) {
  drop_iteration_graph(c);
  free_all(c->bufs.allocs);
  free_all(c->run_allocs);
  c->bufs = Buffers();
  for (auto &p : c->home0)
    p = nullptr;
  c->d_models = nullptr;
  c->d_live = c->d_live_tmp = c->d_gather = c->d_evict = nullptr;
  c->d_gram = c->d_lambda = nullptr;
  c->d_pref = nullptr;
  c->d_wide = nullptr;
  c->d_active = nullptr;
  for (int n = 0; n < CALS_MAX_MODES; n++)
    c->ls_prev[n] = c->ls_backup[n] = nullptr;
  c->ls_prev_lambda = c->ls_backup_lambda = c->ls_partial = nullptr;
  c->uploaded = false;
  c->fitted = false;
  c->run_sig.clear();
}

void disconnect_peers(cals_b200_ctx *c) {
  for (int r = 0; r < CALS_MAX_PEERS; r++) {
    if (c->peer_block[r] && c->peer_is_ipc[r])
      cudaIpcCloseMemHandle(c->peer_block[r]);
    c->peer_block[r] = nullptr;
    c->peer_is_ipc[r] = false;
  }
  c->comm_connected = false;
}

void release_comm(cals_b200_ctx *c) {
  disconnect_peers(c);
  if (c->xblock)
    cudaFree(c->xblock);
  c->xblock = nullptr;
  c->xcap = 0;
  c->comm_connected = false;
  c->comm_rank = 0;
  c->comm_world = 1;
}

void release_corcon(cals_b200_ctx *c) {
  auto &w = c->cc_ws;
  for (int n = 0; n < CALS_MAX_MODES; n++) {
    cudaFree(w.F[n]);
    cudaFree(w.P[n]);
  }
  cudaFree(w.T);
  cudaFree(w.chain[0]);
  cudaFree(w.chain[1]);
  cudaFree(w.tables);
  cudaFree(w.st);
  cudaFree(w.cc);
  cudaFree(w.status);
  cudaFree(w.fail);
  w = cals_b200_ctx::CorconWs();
}

void release_tensor(cals_b200_ctx *c) {
  release_run(c);
  release_corcon(c);
  if (c->Xt && c->Xt != c->Xp)
    cudaFree(c->Xt);
  if (c->Xp)
    cudaFree(c->Xp);
  if (c->jk_norms)
    cudaFree(c->jk_norms);
  if (c->Xq)
    cudaFree(c->Xq);
  if (c->Xr)
    cudaFree(c->Xr);
  c->Xp = c->Xt = c->Xq = c->Xr = c->jk_norms = nullptr;
  c->have_tensor = false;
}

// `modes` are the extents of the whole problem.  slice_mode >= 0: `src` holds only the slab [lo, hi) of that mode
// (dense, same layout, extent hi - lo along slice_mode); the factors keep their full extents.
int install_tensor(cals_b200_ctx *c, int n_modes, const uint64_t *modes, const double *src, bool src_on_device,
                   int slice_mode = -1, long long lo = 0, long long hi = 0) {
  if (n_modes < 3 || n_modes > CALS_MAX_MODES)
    return fail(c, "n_modes must be in [3, %d], got %d", CALS_MAX_MODES, n_modes);
  for (int n = 0; n < n_modes; n++)
    if (modes[n] < 1 || modes[n] > (1u << 30))
      return fail(c, "mode %d has unsupported extent %llu", n, (unsigned long long)modes[n]);
  if (slice_mode >= n_modes)
    return fail(c, "slice_mode %d out of range", slice_mode);
  if (slice_mode >= 0 && (lo < 0 || hi <= lo || hi > (long long)modes[slice_mode] || (lo & 1)))
    return fail(c, "slab [%lld, %lld) of mode %d is empty, out of range or starts at an odd row", lo, hi, slice_mode);
  int xd[CALS_MAX_MODES], roff[CALS_MAX_MODES];
  for (int n = 0; n < n_modes; n++) {
    xd[n] = (n == slice_mode) ? (int)(hi - lo) : (int)modes[n];
    roff[n] = (n == slice_mode) ? (int)lo : 0;
  }
  // same shape as the resident tensor: keep every allocation (and the TMA descriptors that point into them)
  bool same = c->have_tensor && c->geo.n_modes == n_modes;
  for (int n = 0; same && n < n_modes; n++)
    same = c->geo.dims[n] == (int)modes[n] && c->xd[n] == xd[n] && c->roff[n] == roff[n];
  if (!same)
    release_tensor(c);
  long long nX = 1;
  for (int n = 0; n < n_modes; n++) {
    c->geo.dims[n] = (int)modes[n];
    c->geo.ldF[n] = round_up_int((int)modes[n], 2);
    c->xd[n] = xd[n];
    c->roff[n] = roff[n];
    nX *= (long long)xd[n];
  }
  c->geo.n_modes = n_modes;
  c->slice_mode = slice_mode;
  c->nX = nX;
  const int I0 = c->xd[0], I1 = c->xd[1];
  c->ldX0 = round_up_int(I0, 2);
  c->ldX1 = round_up_int(I1, 2);
  const long long rest0 = nX / I0, rest2 = nX / ((long long)I0 * I1);
  c->have_tensor = false;

  double *dense = nullptr;
  if (src_on_device) {
    dense = const_cast<double *>(src);
  } else if (c->ldX0 == I0) {
    // the upload lands directly in Xp
  } else {
    // odd fastest extent: the dense upload goes to a staging block that is kept from call to call (no allocation, no
    // synchronisation on the upload path) and is padded into Xp by a kernel
    if (c->x_stage_cap < (size_t)nX) {
      if (c->x_stage) {
        CU_TRY(c, cudaStreamSynchronize(c->stream));
        cudaFree(c->x_stage);
      }
      c->x_stage = nullptr;
      c->x_stage_cap = 0;
      CU_TRY(c, cudaMalloc((void **)&c->x_stage, (size_t)nX * 8));
      c->x_stage_cap = (size_t)nX;
    }
    dense = c->x_stage;
    CU_TRY(c, cudaMemcpyAsync(dense, src, (size_t)nX * 8, cudaMemcpyHostToDevice, c->stream));
  }
  if (!c->Xp)
    CU_TRY(c, cudaMalloc((void **)&c->Xp, (size_t)c->ldX0 * rest0 * 8));
  if (!src_on_device && c->ldX0 == I0) {
    CU_TRY(c, cudaMemcpyAsync(c->Xp, src, (size_t)nX * 8, cudaMemcpyHostToDevice, c->stream));
    dense = c->Xp;
  } else if (c->ldX0 == I0) {
    CU_TRY(c, cudaMemcpyAsync(c->Xp, dense, (size_t)nX * 8, cudaMemcpyDeviceToDevice, c->stream));
  } else {
    pad_copy_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(dense, c->Xp, I0, c->ldX0, rest0);
  }
  if (!c->Xt)
    CU_TRY(c, cudaMalloc((void **)&c->Xt, (size_t)c->ldX1 * I0 * rest2 * 8));
  {
    dim3 grid((I0 + 31) / 32, (I1 + 31) / 32, (unsigned)std::min<long long>(rest2, 65535));
    swap01_copy_kernel<<<grid, 256, 0, c->stream>>>(dense, c->Xt, I0, I1, c->ldX1, rest2);
  }
  if (n_modes == 4 && slice_mode < 0) { // third layout, for the pair node of modes (0,1) (pairnode.cuh)
    const int I2 = c->xd[2], I3 = c->xd[3];
    c->ldXq = round_up_int(I2, 2);
    if (!c->Xq)
      CU_TRY(c, cudaMalloc((void **)&c->Xq, (size_t)c->ldXq * I3 * I0 * I1 * 8));
    dim3 grid((I0 + 31) / 32, (I2 + 31) / 32, (unsigned)std::min<long long>((long long)I1 * I3, 65535));
    halves_swap_kernel<<<grid, 256, 0, c->stream>>>(c->Xp, c->Xq, I0, I1, I2, I3, c->ldX0, c->ldXq);
  }
  if (c->Xr && build_xr(c)) // same shape as before: the (2, 0, 1) copy that an earlier run made follows the new values
    return 1;
  // norms: one pass over Xp
  if (!c->jk_norms)
    CU_TRY(c, cudaMalloc((void **)&c->jk_norms, (size_t)(I0 + 1) * 8));
  c->d_norm = c->jk_norms + I0;
  {
    const int ctas = (int)std::min<long long>(std::max<long long>(rest0 / 4, 1), (long long)c->sm_count * 4);
    if (c->norm_partial_cap < (size_t)ctas * I0) {
      if (c->norm_partial)
        cudaFree(c->norm_partial);
      c->norm_partial = nullptr;
      CU_TRY(c, cudaMalloc((void **)&c->norm_partial, (size_t)ctas * I0 * 8));
      c->norm_partial_cap = (size_t)ctas * I0;
    }
    rowsumsq_partial_kernel<<<ctas, 256, 256 * 8, c->stream>>>(c->Xp, I0, c->ldX0, rest0, c->norm_partial);
    rowsumsq_final_kernel<<<1, 256, 0, c->stream>>>(c->norm_partial, ctas, I0, c->jk_norms, c->d_norm);
    // no synchronisation here: the upload and the layout kernels overlap with whatever the caller does next (queueing
    // models); the host copy of the norm is picked up by the first call that synchronises anyway
    if (!c->h_norm)
      CU_TRY(c, cudaHostAlloc((void **)&c->h_norm, 64, cudaHostAllocDefault));
    CU_TRY(c, cudaMemcpyAsync(c->h_norm, c->d_norm, 8, cudaMemcpyDeviceToHost, c->stream));
    c->x_norm_valid = false;
    c->x_norm_override = false;
  }
  CU_TRY(c, cudaGetLastError());
  c->have_tensor = true;
  return 0;
}

int ensure_host_norm(cals_b200_ctx *c) {
  if (!c->x_norm_valid) {
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    c->x_norm = *c->h_norm;
    c->x_norm_valid = true;
  }
  return 0;
}

// Shared-memory layout of model_update_kernel for rank R, extent `rows` and the given update method; false when rank R
// does not fit.  The one place that knows the kernel's budget: run_loop sizes the launch with it and
// narrow_rank_bound() derives the largest rank the kernel accepts from it.
struct UpdateSmemPlan {
  int nnls_warps, chunk_rows, table_off;
  size_t smem;
};
bool plan_update_smem(int R, int rows, bool nnls, UpdateSmemPlan *pl) {
  const int R8 = round_up_int(R, 8); // the small matrices and the staged chunk are zero-padded to a multiple of 8
  size_t fixed = ((size_t)2 * R8 * R8 + 4 * R + 64 + 2 * STAT_SEGS * R) * 8; // H / L, block inverses / Gramian,
  // column statistics, 1 / diag(L), diag(H), reduction scratch, statistics candidates
  const size_t budget = 200 * 1024;
  pl->nnls_warps = 0;
  if (nnls) { // per working warp: 5R + R*R doubles and 2R + 1 ints of scratch
    const size_t per_warp = ((size_t)5 * R + (size_t)R * R + (size_t)(2 * R + 2) / 2 + 1) * 8;
    int nw = UPDATE_THREADS / 32;
    while (nw > 1 && fixed + nw * per_warp + (size_t)36 * R8 * 8 > budget)
      nw >>= 1;
    pl->nnls_warps = nw;
    fixed += nw * per_warp;
  }
  if (fixed + (size_t)36 * R8 * 8 > budget)
    return false;
  int cr = round_up_int(rows, 32);
  // behind the staged chunk: tile lookup tables of the fused reduction, (R + chunk rows) ints
  auto tables = [&](int rows_) { return (size_t)((R + rows_ + 1) / 2 + 1) * 8; };
  while (cr >= 32 && fixed + (size_t)(cr + 4) * R8 * 8 + tables(cr) > budget)
    cr -= 32;
  if (cr < 32)
    return false;
  pl->chunk_rows = cr;
  pl->table_off = (int)((fixed + (size_t)(cr + 4) * R8 * 8) / 8);
  pl->smem = fixed + (size_t)(cr + 4) * R8 * 8 + tables(cr);
  return true;
}

// Largest rank the shared-memory update kernel accepts (96 unconstrained, 80 NNLS); models above it are "wide" and
// take the multi-CTA path of wide.cuh (unconstrained only).  The fit does not depend on the extent: a long mode only
// shortens the staged chunk, down to 32 rows.
int narrow_rank_bound(bool nnls) {
  auto largest = [](bool nn) {
    UpdateSmemPlan pl;
    int r = 0;
    while (plan_update_smem(r + 1, 1, nn, &pl))
      r++;
    return r;
  };
  static const int bound[2] = {largest(false), largest(true)}; // thread-safe one-time initialisation
  return bound[nnls ? 1 : 0];
}

// NNLS keeps the rank bound: its row-wise active-set solver needs R^2 scratch per warp in shared memory.
int check_nnls_rank(cals_b200_ctx *c, int model, int rank) {
  const int bound = narrow_rank_bound(true);
  if ((c->flags & CALS_B200_NNLS) && rank > bound)
    return fail(c, "model %d has rank %d, above %d, the largest rank the NNLS update supports", model, rank, bound);
  return 0;
}

// Upload the queued models and allocate every run-time structure.
int prepare_run(cals_b200_ctx *c) {
  if (!c->have_tensor)
    return fail(c, "no tensor set");
  c->fitted = false; // the home matrices are overwritten with the initial factors below
  if (c->hmodels.empty())
    return fail(c, "model queue is empty");
  const Geom &geo = c->geo;
  const int N = geo.n_modes, M = (int)c->hmodels.size();

  // allocation signature: everything below is sized by (dims, buffer_cols, rank sequence)
  std::vector<int> sig;
  sig.reserve((size_t)M + N + 2);
  sig.push_back(N);
  for (int n = 0; n < N; n++) {
    sig.push_back(geo.dims[n]);
    sig.push_back(c->xd[n]);
    sig.push_back(c->roff[n]);
  }
  sig.push_back(c->buffer_cols);
  sig.push_back(c->ls_enabled ? 1 + c->ls_method : 0);
  sig.push_back(c->pair_node);
  sig.push_back(fused_leaf_knob());
  sig.push_back(msdt_knob());
  for (int m = 0; m < M; m++)
    sig.push_back(c->hmodels[m].rank);
  const bool reuse = !c->run_sig.empty() && sig == c->run_sig && c->d_models && c->bufs.cols == c->buffer_cols;
  if (!reuse) {
    release_run(c);
    c->alloc_generation++;
  }

  c->hdesc.assign(M, ModelDesc{});
  const int bound = narrow_rank_bound(false);
  int col = 0, max_rank = 0, narrow_rank = 0, n_wide = 0, wide_min = 0, wide_max = 0;
  long long goff = 0, aoff = 0, sum_rows = 0;
  for (int n = 0; n < N; n++)
    sum_rows += geo.dims[n];
  for (int m = 0; m < M; m++) {
    const HostModel &hm = c->hmodels[m];
    if (hm.rank > c->buffer_cols)
      return fail(c, "model %d has rank %d > buffer_size %d: it can never be admitted", m, hm.rank, c->buffer_cols);
    ModelDesc &d = c->hdesc[m];
    d.rank = hm.rank;
    if (hm.home_col != col)
      return fail(c, "internal error: queue staging out of step");
    d.home_col = col;
    d.jk_mode = hm.jk_mode;
    d.jk_fiber = hm.jk_fiber;
    d.gram_off = goff;
    d.act_off = aoff;
    d.state = MODEL_QUEUED;
    col += hm.rank;
    goff += (long long)N * hm.rank * hm.rank;
    aoff += sum_rows * hm.rank;
    max_rank = std::max(max_rank, hm.rank);
    if (check_nnls_rank(c, m, hm.rank))
      return 1;
    if (hm.rank > bound) {
      wide_min = n_wide ? std::min(wide_min, hm.rank) : hm.rank;
      wide_max = std::max(wide_max, hm.rank);
      n_wide++;
    } else
      narrow_rank = std::max(narrow_rank, hm.rank);
  }
  c->total_cols = col;
  c->max_rank = max_rank;
  c->narrow_rank = narrow_rank;
  c->n_wide = n_wide;
  c->wide_min_rank = wide_min;
  c->wide_max_rank = wide_max;
  c->gram_doubles = goff;
  c->active_bytes = aoff;
  if ((long long)c->h_active.size() != aoff)
    c->h_active.assign((size_t)aoff, 1); // fresh models: every constraint active (reference include/ktensor.h:66)

  if (!reuse) {
    if (alloc_buffers(c, c->bufs, c->buffer_cols, true, c->total_cols))
      return 1;
    if (dev_alloc(c, &c->d_models, (size_t)M, c->run_allocs) || dev_alloc(c, &c->d_live, (size_t)M, c->run_allocs) ||
        dev_alloc(c, &c->d_live_tmp, (size_t)M, c->run_allocs) ||
        dev_alloc(c, &c->d_gather, (size_t)c->buffer_cols, c->run_allocs) ||
        dev_alloc(c, &c->d_evict, (size_t)c->buffer_cols, c->run_allocs) ||
        dev_alloc(c, &c->d_gram, (size_t)goff, c->run_allocs) ||
        dev_alloc(c, &c->d_active, (size_t)aoff, c->run_allocs) ||
        dev_alloc(c, &c->d_lambda, (size_t)c->total_cols, c->run_allocs))
      return 1;
    for (int n = 0; n < N; n++)
      if (dev_alloc(c, &c->home0[n], (size_t)geo.ldF[n] * c->total_cols, c->run_allocs))
        return 1;
    {
      const long long ld8 = round_up_int(std::max(narrow_rank, 1), 8); // wide models never take the prefactor branch
      c->pref_stride = 2 * ld8 * ld8 + 2 * ld8 + 2;
      if (dev_alloc(c, &c->d_pref, (size_t)std::min(M, c->buffer_cols) * (size_t)c->pref_stride, c->run_allocs))
        return 1;
    }
    c->wide_slots = 0;
    if (n_wide > 0) { // one workspace slot per wide model that can be live at the same time
      int max_dim = 0;
      for (int n = 0; n < N; n++)
        max_dim = std::max(max_dim, geo.dims[n]);
      c->wide_ldw = round_up_int(wide_max, WIDE_NB);
      c->wide_y_rows = round_up_int(max_dim, WIDE_NB);
      const long long ldw = c->wide_ldw;
      c->wide_slot_stride = 3 * ldw * ldw + (long long)c->wide_y_rows * ldw + 2 * ldw;
      c->wide_slots = std::min(n_wide, c->buffer_cols / wide_min);
      if (dev_alloc(c, &c->d_wide, (size_t)c->wide_slots * (size_t)c->wide_slot_stride, c->run_allocs))
        return 1;
    }
    if (c->ls_enabled) {
      for (int n = 0; n < N; n++) {
        if (dev_alloc(c, &c->ls_prev[n], (size_t)geo.ldF[n] * c->total_cols, c->run_allocs))
          return 1;
        if (c->ls_method == 0 && dev_alloc(c, &c->ls_backup[n], (size_t)geo.ldF[n] * c->total_cols, c->run_allocs))
          return 1;
      }
      if (dev_alloc(c, &c->ls_prev_lambda, (size_t)c->total_cols, c->run_allocs) ||
          dev_alloc(c, &c->ls_backup_lambda, (size_t)c->total_cols, c->run_allocs) ||
          dev_alloc(c, &c->ls_partial, (size_t)std::min(M, c->buffer_cols) * LS_CHUNKS, c->run_allocs))
        return 1;
    }
  }
  if (ensure_dummy_state(c))
    return 1;

  // upload the initial factors (already in the device layout, pitch ldF, in the pinned input staging)
  for (int n = 0; n < N; n++) {
    const size_t count = (size_t)geo.ldF[n] * c->total_cols;
    if (pinned_reserve(c, &c->h_home[n], &c->h_home_cap[n], count))
      return 1;
    CU_TRY(c, cudaMemcpyAsync(c->bufs.fac.home[n], c->h_in[n], count * 8, cudaMemcpyHostToDevice, c->stream));
    CU_TRY(c, cudaMemcpyAsync(c->home0[n], c->bufs.fac.home[n], count * 8, cudaMemcpyDeviceToDevice, c->stream));
  }
  if (pinned_reserve(c, &c->h_lambda, &c->h_lambda_cap, (size_t)c->total_cols) ||
      pinned_reserve(c, &c->h_desc_pin, &c->h_desc_cap, (size_t)M))
    return 1;
  c->uploaded = true;
  c->run_cols = c->buffer_cols;
  c->run_sig = sig;
  return 0;
}

cudaEvent_t get_event(cals_b200_ctx *c, size_t i) {
  while (c->ev_pool.size() <= i) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    c->ev_pool.push_back(e);
  }
  return c->ev_pool[i];
}

int run_loop(cals_b200_ctx *c, cals_b200_report *rep, bool restore_home) {
  const Geom &geo = c->geo;
  const int N = geo.n_modes, M = (int)c->hmodels.size();
  Buffers &b = c->bufs;
  cudaStream_t s = c->stream;

  // reset device state
  if (restore_home)
    for (int n = 0; n < N; n++)
      CU_TRY(c, cudaMemcpyAsync(b.fac.home[n], c->home0[n], (size_t)geo.ldF[n] * c->total_cols * 8,
                                cudaMemcpyDeviceToDevice, s));
  for (auto &d : c->hdesc) {
    d.state = MODEL_QUEUED;
    d.col = 0;
    d.iters = 0;
    d.chol_info = 0;
    d.error = d.fit = d.old_fit = 0.0;
    d.ls_iter = d.ls_updated_last = d.ls_trial = d.b_iters = 0;
    d.b_error = d.b_fit = d.b_old_fit = 0.0;
  }
  memcpy(c->h_desc_pin, c->hdesc.data(), (size_t)M * sizeof(ModelDesc));
  CU_TRY(c, cudaMemcpyAsync(c->d_models, c->h_desc_pin, (size_t)M * sizeof(ModelDesc), cudaMemcpyHostToDevice, s));
  SchedState st{};
  st.n_models = M;
  st.flags = (int)c->flags;
  st.max_iter = c->max_iter;
  st.buffer_cols = c->buffer_cols;
  st.tol = c->tol;
  st.ls_enabled = c->ls_enabled;
  st.ls_method = c->ls_method;
  st.ls_interval = c->ls_interval;
  st.ls_step = c->ls_step;
  st.x_norm = c->x_norm_valid ? c->x_norm : 0.0;
  st.narrow_on = (c->bufs.narrow && c->variant == CALS_B200_MTTKRP_DMMA) ? 1 : 0;
  CU_TRY(c, cudaMemcpyAsync(c->d_st, &st, sizeof st, cudaMemcpyHostToDevice, s));
  if (!c->x_norm_valid) // set_tensor has not been synchronised yet: take the norm from where the device computed it
    CU_TRY(c, cudaMemcpyAsync(&c->d_st->x_norm, c->d_norm, 8, cudaMemcpyDeviceToDevice, s));
  c->h_flags[0] = c->h_flags[1] = c->h_flags[2] = 0;

  if ((c->flags & CALS_B200_NNLS) && c->active_bytes > 0)
    CU_TRY(c, cudaMemcpyAsync(c->d_active, c->h_active.data(), (size_t)c->active_bytes, cudaMemcpyHostToDevice, s));

  init_grams_kernel<<<dim3(M, N), 256, 0, s>>>(geo, b.fac, c->d_models, c->d_gram);

  SchedParams sp{c->d_st,    c->d_models, c->d_live, c->d_live_tmp,  c->d_gather,
                 c->d_evict, c->d_flags,  b.plans,   c->d_iter_cols};
  const int max_live = std::min(M, c->buffer_cols);
  const dim3 move_grid((c->buffer_cols + MOVE_COLS - 1) / MOVE_COLS, N, 2);

  // The update kernel sums the stream-K partial tiles itself unless the partial result has to leave the device first
  // (sliced tensor), there are no partial tiles (naive variant), or CALS_B200_NO_FUSED_REDUCE=1 asks for the two-kernel
  // path (kept for A/B measurements).
  static const bool fusion_off = getenv("CALS_B200_NO_FUSED_REDUCE") != nullptr;
  // Round 1 used it for small problems (+11 % at 100^3 x 220 columns with the reduce kernel of that time).  With the
  // one-element-per-thread reduce kernel (eight loads in flight, grid over the whole output) the separate pass wins
  // everywhere (config 1: 307.5 k vs 302 k model-iterations/s) -- a few update CTAs cannot pull tens of partial tiles
  // per element as fast as the whole chip -- so the fused form only runs when CALS_B200_FUSED_REDUCE=1 asks for it.
  static const bool fusion_forced = getenv("CALS_B200_FUSED_REDUCE") != nullptr;
  // A wide model's update reads G, so a queue that holds one always runs the separate reduce, which materialises G.
  const bool fused_reduce = c->variant == CALS_B200_MTTKRP_DMMA && !(c->slice_mode >= 0 && c->comm_world > 1) &&
                            !fusion_off && fusion_forced && !b.narrow && c->n_wide == 0;

  // pair nodes: two modes share one contraction of the tensor (pairnode.cuh)
  const bool tree = b.tree && c->variant == CALS_B200_MTTKRP_DMMA;
  auto node_of = [&](int n) { return tree ? b.node_of[n] : -1; };
  // Multi-sweep dimension tree (3 modes, pairnode.cuh): node k contracts mode k and serves modes k+1 and k+2.
  //   even pass:  node 2 (T = X x_2 A_2): mode 0 (first leaf), mode 1 (second leaf);
  //               node 1 (T = X x_1 A_1): mode 2 (first leaf); its second leaf is mode 0 of the NEXT pass
  //   odd pass:   mode 0 from that carried T, or -- when the scheduler moved columns (SchedState::carry_ok == 0) -- from
  //               its own MTTKRP: both sit in the odd iteration body and the one whose turn it is not returns at once;
  //               node 0 (T = X x_0 A_0): mode 1 (first leaf), mode 2 (second leaf)
  // Every mode sees the factors the per-mode MTTKRP sees; three contractions per two passes instead of four.  Pass 0 of
  // every run is even, so nothing is carried into a run.
  const bool msdt = tree && b.msdt && !c->ls_enabled && !fused_reduce;
  // per mode and parity: node whose T serves the mode (-1: its own MTTKRP), whether that T is made right before
  struct Source {
    int node;
    bool contract, carried;
  };
  auto source = [&](int n, int odd) -> Source {
    if (msdt && !odd)
      return {n == 2 ? 1 : 2, n != 1, false};
    if (msdt)
      return {n == 0 ? 1 : 0, n == 1, n == 0};
    const int k = node_of(n);
    return {k, k >= 0 && n == b.node[k].pg.mode_fast, false};
  };

  // tuning aid: CALS_B200_UPDATE_PROF=1 prints the phase times of the update kernel's slowest CTA per mode after the run
  static const bool update_prof = getenv("CALS_B200_UPDATE_PROF") != nullptr;
  if (update_prof && !c->d_update_prof) {
    CU_TRY(c, cudaMalloc((void **)&c->d_update_prof, (size_t)CALS_MAX_MODES * 8192 * 16 * sizeof(long long)));
    CU_TRY(c, cudaMemset(c->d_update_prof, 0, (size_t)CALS_MAX_MODES * 8192 * 16 * sizeof(long long)));
  }
  if (max_live > 8192 && c->d_update_prof) {
    cudaFree(c->d_update_prof);
    c->d_update_prof = nullptr;
  }
  // shared memory of the update kernel
  UpdateParams up[CALS_MAX_MODES];
  size_t up_smem[CALS_MAX_MODES];
  for (int n = 0; n < N; n++) {
    UpdateParams &u = up[n];
    u.mode = n;
    u.n_modes = N;
    u.rows = geo.dims[n];
    u.ld = geo.ldF[n];
    // sized for the largest narrow rank; the CTAs of wide models return at once
    const int R = std::max(c->narrow_rank, 1);
    u.nnls = (c->flags & CALS_B200_NNLS) ? 1 : 0;
    UpdateSmemPlan pl;
    if (!plan_update_smem(R, u.rows, u.nnls, &pl))
      return fail(c, "rank %d too large for the shared-memory update kernel", R);
    const int cr = pl.chunk_rows;
    u.nnls_warps = pl.nnls_warps;
    u.chunk_rows = cr;
    u.chunk_pitch = cr + 4; // = 4 mod 16 doubles: the DMMA fragment loads of the update kernel are bank-conflict free
    u.table_off = pl.table_off;
    u.max_rank = R;
    u.G = b.G;
    u.F[0] = b.fac.buf[0][n];
    u.F[1] = b.fac.buf[1][n];
    u.gram_pool = c->d_gram;
    u.lambda_home = c->d_lambda;
    u.x_norms_jk = c->jk_norms;
    u.models = c->d_models;
    u.live = c->d_live;
    u.st = c->d_st;
    u.act_pool = c->d_active;
    u.plan = (fused_reduce && node_of(n) < 0) ? b.plans.plan[n] : nullptr;
    u.ws = b.ws;
    u.plan_ctas = c->sm_count;
    u.tile_elems = tile_m(b.wm[n]) * TILE_N;
    u.n_tile = TILE_N;
    u.G_out = b.G;
    u.rows_before = 0;
    for (int k = 0; k < n; k++)
      u.rows_before += geo.dims[k];
    u.pref = nullptr;
    u.pref_stride = 0;
    u.prof = c->d_update_prof ? c->d_update_prof + (size_t)n * max_live * 16 : nullptr;
    up_smem[n] = pl.smem;
  }
  // models of rank above the bound: the multi-CTA update of wide.cuh after the narrow one, per mode
  const bool has_wide = c->n_wide > 0;
  const bool has_narrow = c->n_wide < M;
  WideParams wp[CALS_MAX_MODES];
  for (int n = 0; n < N && has_wide; n++) {
    WideParams &w = wp[n];
    w.mode = n;
    w.n_modes = N;
    w.rows = geo.dims[n];
    w.ld = geo.ldF[n];
    w.bound = narrow_rank_bound(false);
    w.G = b.G;
    w.F[0] = b.fac.buf[0][n];
    w.F[1] = b.fac.buf[1][n];
    w.gram_pool = c->d_gram;
    w.lambda_home = c->d_lambda;
    w.x_norms_jk = c->jk_norms;
    w.models = c->d_models;
    w.live = c->d_live;
    w.st = c->d_st;
    w.ws = c->d_wide;
    w.slot_stride = c->wide_slot_stride;
    w.ldw = c->wide_ldw;
    w.y_rows = c->wide_y_rows;
  }
  if (has_wide && !c->wide_attr_done) {
    CU_TRY(c, cudaFuncSetAttribute(wide_factor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)WIDE_FACTOR_SMEM));
    CU_TRY(c, cudaFuncSetAttribute(wide_solve_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)WIDE_TILE_SMEM));
    CU_TRY(c, cudaFuncSetAttribute(wide_solve_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)WIDE_TILE_SMEM));
    CU_TRY(c, cudaFuncSetAttribute(wide_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WIDE_TILE_SMEM));
    c->wide_attr_done = true;
  }
  if ((c->flags & CALS_B200_NNLS) && c->max_rank > narrow_rank_bound(true)) // options changed after prepare_run
    for (int m = 0; m < M; m++)
      if (check_nnls_rank(c, m, c->hmodels[m].rank))
        return 1;
  {
    size_t mx = 0;
    for (int n = 0; n < N; n++)
      mx = std::max(mx, up_smem[n]);
    if (raise_smem_limit(c, (const void *)model_update_kernel<false>, mx) ||
        raise_smem_limit(c, (const void *)model_update_kernel<true>, mx))
      return 1;
  }

  // slab mode over several GPUs: every MTTKRP is followed by the peer-memory exchange (comm.cuh)
  const bool exchange = c->slice_mode >= 0 && c->comm_world > 1;
  CommParams cp{};
  size_t max_ld = 0;
  for (int n = 0; n < N; n++)
    max_ld = std::max<size_t>(max_ld, (size_t)geo.ldF[n]);
  if (exchange) {
    if (!c->comm_connected)
      return fail(c, "the tensor is sliced over %d GPUs but the peers are not connected (cals_b200_comm_connect)",
                  c->comm_world);
    if (max_ld * (size_t)c->buffer_cols > c->xcap)
      return fail(c, "exchange buffers hold %zu doubles, this run needs %zu (cals_b200_comm_alloc capacity)", c->xcap,
                  max_ld * (size_t)c->buffer_cols);
    cp.rank = c->comm_rank;
    cp.world = c->comm_world;
    cp.slice_mode = c->slice_mode;
    for (int r = 0; r <= c->comm_world; r++)
      cp.cuts[r] = c->cuts[r];
    for (int r = 0; r < c->comm_world; r++) {
      cp.peer_flags[r] = (unsigned long long *)c->peer_block[r];
      cp.peer_x[r] = (const double *)((char *)c->peer_block[r] + COMM_FLAG_BYTES);
    }
    cp.cap = c->xcap;
    cp.seq_base = c->seq_base;
    cp.spin_limit = 40000000000ll; // ~20 s at 1.97 GHz: a peer that has not arrived by then is gone
  }

  LsParams lp{};
  if (c->ls_enabled) {
    if (c->slice_mode >= 0 && c->comm_world > 1 && c->ls_method != 0)
      return fail(c, "line search with error checking needs the whole tensor on one GPU");
    if (c->flags & CALS_B200_NNLS)
      return fail(c, "line search together with the NNLS update is not supported");
    lp.geo = geo;
    lp.fac = b.fac;
    for (int n = 0; n < N; n++) {
      lp.prev[n] = c->ls_prev[n];
      lp.backup[n] = c->ls_backup[n];
    }
    lp.prev_lambda = c->ls_prev_lambda;
    lp.backup_lambda = c->ls_backup_lambda;
    lp.lambda_home = c->d_lambda;
    lp.gram_pool = c->d_gram;
    lp.models = c->d_models;
    lp.live = c->d_live;
    lp.st = c->d_st;
    lp.X = c->Xp;
    lp.ldX0 = c->ldX0;
    lp.rest0 = c->nX / c->xd[0];
    lp.partial = c->ls_partial;
    lp.chunks = LS_CHUNKS;
  }

  const int RA = 4; // host run-ahead in CALS iterations
  cudaEvent_t ring[RA];
  for (int i = 0; i < RA; i++)
    ring[i] = get_event(c, i);
  cudaEvent_t ev_begin = get_event(c, RA), ev_end = get_event(c, RA + 1);
  size_t ev_next = RA + 2;
  // per-kernel timing (cals_b200_set_timing): windows between events recorded on the stream
  enum { T_MTTKRP = 0, T_UPDATE = 1, T_EXCHANGE = 2, T_PAIR_GEMM = 3, T_PAIR_LEAF = 4 };
  struct Window {
    size_t e0, e1;
    int kind;
    long long iteration;
    int odd; // parity of the iteration body that recorded it
  };
  std::vector<Window> timed;
  int body_odd = 0; // parity of the iteration body being enqueued

  uint64_t launches = 1, mttkrp_launches = 0;
  auto t0 = std::chrono::steady_clock::now();
  CU_TRY(c, cudaEventRecord(ev_begin, s));
  long long it = 0;
  bool capturing_timed = false;
  auto mark = [&]() -> size_t { // no-op unless timing is on
    if (!c->timing)
      return 0;
    // inside a stream capture only an EXTERNAL record becomes an event-record node of the graph (a plain record is
    // an internal fork / join dependency and never fires at replay)
    if (capturing_timed)
      cudaEventRecordWithFlags(get_event(c, ev_next), s, cudaEventRecordExternal);
    else
      cudaEventRecord(get_event(c, ev_next), s);
    return ev_next++;
  };
  auto window = [&](size_t e0, size_t e1, int kind) {
    if (c->timing)
      timed.push_back({e0, e1, kind, it, body_odd});
  };
  // everything one CALS iteration launches, in stream order; odd: the odd body of the multi-sweep schedule
  int launches_per_iteration[2] = {0, 0};
  bool pref_on = false; // decided below, before the first call of enqueue_iteration
  auto enqueue_iteration = [&](bool count, int odd) -> int {
    int n_launch = 0;
    body_odd = odd;
    auto chain_ok = [&](cudaError_t e, const char *what) {
      if (e != cudaSuccess)
        fail(c, "launch of %s failed: %s", what, cudaGetErrorString(e));
      return e == cudaSuccess;
    };
    SchedParams spi = sp;
    spi.carry = msdt && odd;
    spi.contractions = 0; // (the fallback MTTKRP of an odd pass is counted by the scheduler itself)
    for (int n = 0; n < N; n++) {
      const Source src = source(n, odd);
      spi.contractions += (src.node < 0 || src.contract) ? 1 : 0;
    }
    sched_kernel<<<1, 32, 0, s>>>(spi); // first kernel of the iteration: plain stream order after the previous iteration
    if (!chain_ok(launch_chain(c, move_kernel, move_grid, dim3(256), (size_t)0, geo, b.fac, (const SchedState *)c->d_st,
                               (const int *)c->d_gather, (const int *)c->d_evict),
                  "move_kernel"))
      return -1;
    n_launch += 2;
    if (c->ls_enabled) {
      ls_snapshot_kernel<<<max_live, 256, 0, s>>>(lp);
      n_launch++;
    }
    for (int n = 0; n < N; n++) {
      const size_t e0 = mark();
      size_t e1;
      const Source src = source(n, odd);
      if (src.node >= 0) {
        const Buffers::PairNode &nd = b.node[src.node];
        size_t el = e0;
        if (src.contract) { // first mode served by this T: make it
          if (nd.slot < 0) {
            if (launch_pair_gemm(c, b, src.node))
              return -1;
            n_launch += b.narrow ? 2 : 1;
          } else {
            if (launch_mttkrp(c, b, nd.slot, 0, c->variant, false, false, nd.T))
              return -1;
            n_launch += b.narrow ? 3 : 2;
          }
          el = mark();
          window(e0, el, T_PAIR_GEMM);
        }
        if (pref_on) { // the update's Cholesky runs on a forked branch next to the leaf that streams T
          if (fork_prefactor(c, n))
            return -1;
          n_launch++;
        }
        if (launch_pair_leaf(c, b, src.node, n, exchange, src.carried))
          return -1;
        n_launch++;
        if (exchange) {
          const size_t x0 = mark();
          exchange_sum_kernel<<<c->sm_count * 2, 256, 0, s>>>(cp, c->d_st, b.G, n, N, geo.dims[n], geo.ldF[n]);
          window(x0, mark(), T_EXCHANGE);
          n_launch++;
        }
        e1 = mark();
        window(el, e1, T_PAIR_LEAF); // includes the exchange
        if (src.carried) { // ... or, when the columns moved, mode 0's own MTTKRP (no exchange: the tensor is whole here)
          if (launch_mttkrp(c, b, n, 0, c->variant, false, false, nullptr, true))
            return -1;
          n_launch += 2;
          const size_t e2 = mark();
          window(e1, e2, T_MTTKRP);
          e1 = e2;
        }
      } else {
        if (pref_on) { // ... or next to the partial-tile reduction (launch_dmma forks between its two kernels)
          if (c->variant == CALS_B200_MTTKRP_NAIVE) {
            if (fork_prefactor(c, n))
              return -1;
          } else
            c->fork_mode = n;
          n_launch++;
        }
        if (launch_mttkrp(c, b, n, 0, c->variant, exchange, fused_reduce))
          return -1;
        c->fork_mode = -1;
        n_launch += (c->variant == CALS_B200_MTTKRP_NAIVE || fused_reduce) ? 1 : (b.narrow ? 3 : 2);
        if (exchange) {
          const size_t x0 = mark();
          exchange_sum_kernel<<<c->sm_count * 2, 256, 0, s>>>(cp, c->d_st, b.G, n, N, geo.dims[n], geo.ldF[n]);
          window(x0, mark(), T_EXCHANGE);
          n_launch++;
        }
        e1 = mark();
        window(e0, e1, T_MTTKRP); // includes the exchange
      }
      if (pref_on && join_prefactor(c, n))
        return -1;
      if (has_narrow) {
        if (!chain_ok(up[n].nnls ? launch_chain(c, model_update_kernel<true>, dim3(max_live), dim3(UPDATE_THREADS),
                                                up_smem[n], up[n])
                                 : launch_chain(c, model_update_kernel<false>, dim3(max_live), dim3(UPDATE_THREADS),
                                                up_smem[n], up[n]),
                      "model_update_kernel"))
          return -1;
        n_launch++;
      }
      if (has_wide) {
        const int S = c->wide_slots, CT = c->wide_ldw / WIDE_NB, RT = (geo.dims[n] + WIDE_NB - 1) / WIDE_NB;
        wide_factor_kernel<<<dim3(WIDE_CLUSTER, S), WIDE_THREADS, WIDE_FACTOR_SMEM, s>>>(wp[n]);
        wide_solve_kernel<0><<<dim3(RT * CT, S), WIDE_THREADS, WIDE_TILE_SMEM, s>>>(wp[n]);
        wide_solve_kernel<1><<<dim3(RT * CT, S), WIDE_THREADS, WIDE_TILE_SMEM, s>>>(wp[n]);
        wide_stats_kernel<<<dim3(c->wide_ldw / WIDE_STAT_COLS, S), WIDE_THREADS, 0, s>>>(wp[n]);
        wide_gram_kernel<<<dim3(CT * (CT + 1) / 2, S), WIDE_THREADS, WIDE_TILE_SMEM, s>>>(wp[n]);
        n_launch += 5;
        if (n == N - 1) {
          wide_error_kernel<<<S, WIDE_THREADS, 0, s>>>(wp[n]);
          n_launch++;
        }
        if (!chain_ok(cudaGetLastError(), "the wide-model update kernels"))
          return -1;
      }
      window(e1, mark(), T_UPDATE);
    }
    if (c->ls_enabled) {
      ls_main_kernel<<<max_live, 256, 0, s>>>(lp);
      n_launch++;
      if (c->ls_method != 0) {
        ls_explicit_error_kernel<<<dim3(max_live, LS_CHUNKS), 256, (size_t)(c->max_rank + 32) * 8, s>>>(lp);
        ls_decide_kernel<<<max_live, 256, 0, s>>>(lp);
        n_launch += 2;
      }
    }
    if (count)
      launches_per_iteration[odd] = n_launch;
    return n_launch;
  };

  // Graph mode (default): capture the iteration once, replay it.  Off with per-kernel timing (events sit between the
  // kernels), with the sliced-tensor exchange (its sequence base changes from run to run) and with CALS_B200_NO_GRAPH=1.
  static const bool graphs_off = getenv("CALS_B200_NO_GRAPH") != nullptr;
  const bool use_graph = !c->timing && !exchange && !graphs_off;
  // Programmatic dependent launch between the kernels of the chain: OFF unless CALS_B200_PDL=1.  Measured on the B200
  // inside the replayed graph it costs throughput on every configuration (config 2: 85.3 k -> 82.4 k, its 8-way shard
  // 52.7 k -> 48.1 k, config 1: 302 k -> 291 k model-iterations/s): the early-scheduled CTAs of the next kernel hold
  // shared memory and registers on the SMs the running kernel still uses, and graph kernel nodes already launch
  // back to back.  Never used with per-kernel timing, line search or the sliced-tensor exchange.
  static const int graph_batch = [] { // CALS iterations per graph launch when the pass count is known (tuning knob)
    const char *e = getenv("CALS_B200_GRAPH_BATCH");
    const int v = e ? atoi(e) : 5;
    return v < 1 ? 1 : (v > 64 ? 64 : v);
  }();
  static const bool pdl_on = getenv("CALS_B200_PDL") != nullptr;
  c->pdl = use_graph && pdl_on && !c->ls_enabled;
  // function attributes must be set outside of a capture: launch_dmma does it lazily, so trigger it here
  auto prepare_capture = [&]() -> int {
    for (int n = 0; n < N; n++)
      if (c->variant == CALS_B200_MTTKRP_DMMA && ensure_dmma_attr(c, b.wm[n]))
        return 1;
    for (int k = 0; tree && k < b.n_nodes; k++)
      if (b.node[k].slot < 0 ? launch_pair_gemm(c, b, k, true) : ensure_dmma_attr(c, b.wm[b.node[k].slot]))
        return 1;
    return 0;
  };
  // Per-kernel timing inside a graph: the events between the kernels are captured as event-record nodes of a
  // one-iteration graph, which is replayed pass by pass with a synchronisation (and a read of the windows) after each.
  // The kernels then follow each other as closely as in the untimed replay; with plain stream launches every event and
  // every launch adds microseconds of idle time, which inflates the windows of short kernels (a 140 us contraction of an
  // 8-way shard was reported as 175 us).
  const bool timed_graph = c->timing && !exchange && !graphs_off && !c->ls_enabled;
  cudaGraphExec_t tgraph[2] = {};
  double tsum[5] = {0, 0, 0, 0, 0};
  const int n_bodies = msdt ? 2 : 1; // iteration bodies: even (and odd)
  // The head of every update (H, Cholesky, block inverses) on a forked branch of the iteration graph, off the critical
  // path (update.cuh: prefactor_kernel).  OFF unless CALS_B200_PREFACTOR=1: measured on the B200 the fork / join edges
  // and the kernel running next to the leaf cost more than the 17 k cycles they take out of the update kernel (8-way
  // shard of config 2: 56.7 k -> 54.0 k model-iterations/s, the leaf beside it 25 -> 31 us; config 1 +0.6 %, config 2 0).
  static const bool pref_wanted = getenv("CALS_B200_PREFACTOR") != nullptr;
  pref_on = (use_graph || timed_graph) && pref_wanted && !(c->flags & CALS_B200_NNLS) && !c->ls_enabled && !fused_reduce &&
            c->d_pref != nullptr;
  {
    const long long ld8 = round_up_int(std::max(c->narrow_rank, 1), 8);
    c->pf_smem = (size_t)(2 * ld8 * ld8 + 2 * ld8) * 8;
    c->pf_grid = max_live;
    if (pref_on && c->pf_smem > 200 * 1024)
      pref_on = false;
    if (pref_on && raise_smem_limit(c, (const void *)prefactor_kernel, c->pf_smem))
      return 1;
    for (int n = 0; n < N; n++) {
      PrefactorParams &q = c->pf[n];
      q.mode = n;
      q.n_modes = N;
      q.gram_pool = c->d_gram;
      q.models = c->d_models;
      q.live = c->d_live;
      q.st = c->d_st;
      q.pref = c->d_pref;
      q.pref_stride = c->pref_stride;
      q.max_rank = std::max(c->narrow_rank, 1);
      up[n].pref = pref_on ? c->d_pref : nullptr;
      up[n].pref_stride = c->pref_stride;
    }
  }
  auto free_tgraphs = [&]() {
    for (auto &g : tgraph)
      if (g)
        cudaGraphExecDestroy(g);
  };
  if (timed_graph) {
    if (prepare_capture())
      return 1;
    // create the events of the iteration bodies before the capture begins
    get_event(c, ev_next + 16 * (size_t)(N + 2) * n_bodies);
    for (int odd = 0; odd < n_bodies; odd++) {
      cudaGraph_t graph = nullptr;
      CU_TRY(c, cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
      capturing_timed = true;
      const int rc = enqueue_iteration(true, odd);
      capturing_timed = false;
      cudaError_t ce = cudaStreamEndCapture(s, &graph);
      if (rc < 0 || ce != cudaSuccess) {
        if (graph)
          cudaGraphDestroy(graph);
        free_tgraphs();
        return rc < 0 ? 1 : fail(c, "cudaStreamEndCapture (timed) failed: %s", cudaGetErrorString(ce));
      }
      ce = cudaGraphInstantiate(&tgraph[odd], graph, 0);
      cudaGraphDestroy(graph);
      if (ce != cudaSuccess) {
        free_tgraphs();
        return fail(c, "cudaGraphInstantiate (timed) failed: %s", cudaGetErrorString(ce));
      }
    }
  }
  if (use_graph) {
    std::vector<long long> key = {c->alloc_generation, (long long)c->flags, c->ls_enabled, c->ls_method, c->variant,
                                  (long long)max_live, fused_reduce ? 1 : 0, tree ? 1 : 0, c->pdl ? 1 : 0, graph_batch,
                                  pref_on ? 1 : 0, msdt ? 1 : 0};
    const bool same_graph = c->iter_graph[0] && c->iter_graph_key.size() == key.size() + 2 &&
                            std::equal(key.begin(), key.end(), c->iter_graph_key.begin());
    if (!same_graph) {
      drop_iteration_graph(c);
      if (prepare_capture())
        return 1;
      // per body parity, two graphs: one CALS iteration, and GRAPH_BATCH iterations back to back starting with that
      // parity (used while the number of passes still to run is known to be at least that, see below)
      for (int odd = 0; odd < n_bodies; odd++)
        for (int which = 0; which < 2; which++) {
          cudaGraph_t graph = nullptr;
          CU_TRY(c, cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
          int rc = 0;
          for (int k = 0; k < (which == 0 ? 1 : graph_batch) && rc >= 0; k++)
            rc = enqueue_iteration(true, msdt ? (odd + k) & 1 : 0);
          cudaError_t ce = cudaStreamEndCapture(s, &graph);
          if (rc < 0 || ce != cudaSuccess) {
            if (graph)
              cudaGraphDestroy(graph);
            return rc < 0 ? 1 : fail(c, "cudaStreamEndCapture failed: %s", cudaGetErrorString(ce));
          }
          ce = cudaGraphInstantiate(which == 0 ? &c->iter_graph[odd] : &c->batch_graph[odd], graph, 0);
          cudaGraphDestroy(graph);
          if (ce != cudaSuccess)
            return fail(c, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ce));
        }
      c->iter_graph_key = key;
      c->iter_graph_key.push_back(launches_per_iteration[0]);
      c->iter_graph_key.push_back(launches_per_iteration[1]);
    } else {
      launches_per_iteration[0] = (int)c->iter_graph_key[key.size()];
      launches_per_iteration[1] = (int)c->iter_graph_key[key.size() + 1];
    }
  }

  // Forced iteration count with the whole queue resident from the first pass (the benchmark protocol, parameter sweeps):
  // the loop runs exactly max_iter + 1 passes (the last one only evicts), so the host can replay batches of passes per
  // graph launch and stop on the dot instead of running RA - 1 empty passes ahead of the `done` flag.
  long long known_passes = -1, n_submits = 0;
  if ((c->flags & CALS_B200_FORCE_MAX_ITER) && !(c->flags & CALS_B200_ALWAYS_EVICT_FIRST) &&
      c->total_cols <= c->buffer_cols && !c->ls_enabled)
    known_passes = (long long)c->max_iter + 1;
  for (;; it++) {
    const int odd = msdt ? (int)(it & 1) : 0; // the host picks the body by the parity of the pass
    if (timed_graph) {
      CU_TRY(c, cudaGraphLaunch(tgraph[odd], s));
      launches += launches_per_iteration[odd];
      mttkrp_launches += N;
      CU_TRY(c, cudaStreamSynchronize(s));
      const bool drained = *(volatile int *)&c->h_flags[0] != 0; // this pass found the queue empty: no work in it
      if (!drained)
        for (auto &t : timed) {
          if (t.odd != odd)
            continue;
          float e = 0;
          cudaEventElapsedTime(&e, get_event(c, t.e0), get_event(c, t.e1));
          tsum[t.kind] += e;
        }
      if (drained)
        break;
      continue;
    }
    if (use_graph && known_passes > 0 && it + graph_batch <= known_passes && graph_batch > 1) {
      CU_TRY(c, cudaGraphLaunch(c->batch_graph[odd], s));
      for (int k = 0; k < graph_batch; k++)
        launches += (uint64_t)launches_per_iteration[msdt ? (odd + k) & 1 : 0];
      mttkrp_launches += (uint64_t)N * (graph_batch - 1);
      it += graph_batch - 1;
    } else if (use_graph) {
      CU_TRY(c, cudaGraphLaunch(c->iter_graph[odd], s));
      launches += launches_per_iteration[odd];
    } else {
      const int rc = enqueue_iteration(false, odd);
      if (rc < 0)
        return 1;
      launches += rc;
    }
    mttkrp_launches += N;
    CU_TRY(c, cudaEventRecord(ring[n_submits % RA], s));
    if (n_submits >= RA - 1)
      CU_TRY(c, cudaEventSynchronize(ring[(n_submits + 1) % RA]));
    n_submits++;
    if (known_passes > 0 && use_graph && it + 1 >= known_passes)
      break; // every pass has been enqueued; the synchronisation below waits for the last one
    if (*(volatile int *)&c->h_flags[0])
      break;
    if (c->timing && ev_next > 100000) {
      return fail(c, "per-kernel timing supports at most ~100000 events per run");
    }
  }
  CU_TRY(c, cudaEventRecord(ev_end, s));
  CU_TRY(c, cudaStreamSynchronize(s));
  CU_TRY(c, cudaGetLastError());
  auto t1 = std::chrono::steady_clock::now();
  free_tgraphs();

  if (update_prof && c->d_update_prof) {
    std::vector<long long> h((size_t)N * max_live * 16);
    cudaMemcpy(h.data(), c->d_update_prof, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
    for (int n = 0; n < N; n++) {
      int worst = 0;
      long long worst_t = -1;
      for (int b2 = 0; b2 < max_live; b2++) {
        const long long *r = &h[((size_t)n * max_live + b2) * 16];
        if (r[9] - r[0] > worst_t) {
          worst_t = r[9] - r[0];
          worst = b2;
        }
      }
      const long long *r = &h[((size_t)n * max_live + worst) * 16];
      fprintf(stderr, "[update prof] mode %d slowest CTA %d rank %lld: H %lld | chol %lld (stage+sync %lld) | solve %lld | "
                      "stats %lld | lambda %lld | scale %lld | gram %lld | publish %lld | tail %lld | total %lld cycles\n",
              n, worst, r[15], r[1] - r[0], r[2] - r[1], r[3] - r[2], r[4] - r[3], r[5] - r[4], r[6] - r[5], r[7] - r[6],
              r[8] - r[7], r[9] - r[8], r[10] ? r[10] - r[9] : 0, (r[10] ? r[10] : r[9]) - r[0]);
    }
  }
  // scalars back
  CU_TRY(c, cudaMemcpy(&st, c->d_st, sizeof st, cudaMemcpyDeviceToHost));
  c->last_global_iter = st.global_iter;
  c->last_ls_performed = st.ls_performed;
  c->last_ls_failed = st.ls_failed;
  if (exchange) {
    c->seq_base += st.global_iter * (unsigned long long)N; // the next run's first exchange continues the sequence
    if (st.comm_error)
      return fail(c, "a peer GPU did not reach an exchange point within the time limit (rank %d of %d)", c->comm_rank,
                  c->comm_world);
  }
  if (rep) {
    memset(rep, 0, sizeof *rep);
    rep->iter = st.global_iter;
    rep->n_ktensors = st.n_admitted;
    rep->ktensor_comp_sum = st.comp_sum;
    if (ensure_host_norm(c))
      return 1;
    rep->x_norm = c->x_norm;
    rep->total_time = std::chrono::duration<double>(t1 - t0).count();
    float ms = 0;
    cudaEventElapsedTime(&ms, ev_begin, ev_end);
    rep->device_ms = ms;
    // Passes launched after the queue drained (host run-ahead) find C == 0 and exit at once: they are real launches
    // (kernel_launches) but not MTTKRP work, so the per-launch statistics only count the st.global_iter real passes.
    const uint64_t real_mttkrp = (uint64_t)st.global_iter * (uint64_t)N;
    rep->mttkrp_launches = real_mttkrp;
    rep->kernel_launches = launches;
    rep->mttkrp_flops = 2.0 * (double)c->nX * (double)N * (double)st.col_iter_sum;
    // flop that actually ran on the tensor cores: the scheduler counts the contractions of every executed pass (pair
    // nodes: two per iteration instead of N; multi-sweep schedule: three per two iterations, plus the fallback MTTKRPs)
    rep->tree = tree ? 1 : 0;
    rep->fused_leaf_blocks = (tree && N == 3 && b.node[0].pg.fuse_slow && !exchange)
                                 ? (b.node[0].pg.E2 + b.node[0].wm - 1) / b.node[0].wm
                                 : 0;
    rep->tensor_flops = 2.0 * (double)c->nX * (double)st.contraction_cols;
    rep->sweep_period = msdt ? 2 : 1;
    if (c->timing) {
      // passes launched after the queue drained (host run-ahead) are not counted
      double sum[5] = {0, 0, 0, 0, 0};
      if (timed_graph) {
        for (int k = 0; k < 5; k++)
          sum[k] = tsum[k];
      } else
        for (auto &t : timed) {
          if (t.iteration >= (long long)st.global_iter)
            continue;
          float e = 0;
          cudaEventElapsedTime(&e, get_event(c, t.e0), get_event(c, t.e1));
          sum[t.kind] += e;
        }
      rep->mttkrp_ms = sum[T_MTTKRP] + sum[T_PAIR_GEMM] + sum[T_PAIR_LEAF];
      rep->update_ms = sum[T_UPDATE];
      rep->exchange_ms = sum[T_EXCHANGE];
      rep->pair_gemm_ms = sum[T_PAIR_GEMM];
      rep->pair_leaf_ms = sum[T_PAIR_LEAF];
    }
  }
  c->results_fresh = false;
  c->fitted = true;
  return 0;
}

int download_results(cals_b200_ctx *c) {
  if (c->results_fresh)
    return 0;
  if (!c->uploaded)
    return fail(c, "no run to fetch results from");
  const Geom &geo = c->geo;
  for (int n = 0; n < geo.n_modes; n++)
    CU_TRY(c, cudaMemcpyAsync(c->h_home[n], c->bufs.fac.home[n], (size_t)geo.ldF[n] * c->total_cols * 8,
                              cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(c, cudaMemcpyAsync(c->h_lambda, c->d_lambda, (size_t)c->total_cols * 8, cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(c, cudaMemcpyAsync(c->h_desc_pin, c->d_models, c->hdesc.size() * sizeof(ModelDesc), cudaMemcpyDeviceToHost,
                            c->stream));
  CU_TRY(c, cudaStreamSynchronize(c->stream));
  memcpy(c->hdesc.data(), c->h_desc_pin, c->hdesc.size() * sizeof(ModelDesc));
  c->results_fresh = true;
  return 0;
}

void copy_model_out(cals_b200_ctx *c, int m, double *const *factors_out, double *lambda_out,
                    cals_b200_model_stats *stats) {
  const Geom &geo = c->geo;
  const ModelDesc &d = c->hdesc[m];
  if (factors_out)
    for (int n = 0; n < geo.n_modes; n++) {
      if (!factors_out[n])
        continue;
      const int rows = geo.dims[n], ld = geo.ldF[n];
      for (int j = 0; j < d.rank; j++)
        memcpy(factors_out[n] + (size_t)j * rows, &c->h_home[n][(size_t)(d.home_col + j) * ld], (size_t)rows * 8);
    }
  if (lambda_out)
    memcpy(lambda_out, &c->h_lambda[d.home_col], (size_t)d.rank * 8);
  if (stats) {
    stats->iters = (uint64_t)d.iters;
    stats->error = d.error;
    stats->fit = d.fit;
    stats->old_fit = d.old_fit;
    stats->chol_info = d.chol_info;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Core consistency of every queued model (corcon.cuh).  Models go in queue order, in batches of whole models; a batch
// holds at most buffer_cols columns, and its T and each of its two chain buffers stay within CC_BATCH_CAP_BYTES (a
// single model may exceed that on its own).
constexpr size_t CC_BATCH_CAP_BYTES = (size_t)2 << 30;
constexpr size_t CC_HEADROOM_BYTES = (size_t)2 << 30; // device memory left free, as for the pair node's T

template <typename T> int cc_grow(cals_b200_ctx *c, T **p, size_t *cap, size_t n) {
  if (*p && *cap >= n)
    return 0;
  cudaFree(*p);
  *p = nullptr;
  *cap = 0;
  CU_TRY(c, cudaMalloc((void **)p, std::max<size_t>(n, 1) * sizeof(T)));
  *cap = n;
  return 0;
}

template <int WM>
int launch_cc_pair_gemm(cals_b200_ctx *c, const PairMaps &maps, const PairGeom &pg, const SchedState *st, double *T) {
  auto kern = pair_gemm_kernel<WM, WN_FIXED>;
  constexpr int smem = PairCfg<WM, WN_FIXED>::SMEM_BYTES;
  if (raise_smem_limit(c, (const void *)kern, smem))
    return 1;
  kern<<<c->sm_count, MTTKRP_THREADS, smem, c->stream>>>(maps, pg, st, T, nullptr);
  CU_TRY(c, cudaGetLastError());
  return 0;
}

int core_consistency(cals_b200_ctx *c, double *cc_out, int32_t *status_out) {
  if (!c->have_tensor)
    return fail(c, "no tensor set");
  const Geom &geo = c->geo;
  const int N = geo.n_modes, M = (int)c->hmodels.size();
  if (N > 4)
    return fail(c, "core consistency supports tensors of 3 and 4 modes, this one has %d", N);
  if (c->slice_mode >= 0)
    return fail(c, "core consistency needs the whole tensor on one device; this context holds a slab of mode %d",
                c->slice_mode);
  if (M == 0)
    return 0;
  cudaStream_t s = c->stream;
  auto &w = c->cc_ws;
  const int *dims = geo.dims;

  // statuses known before any computation: 1 = rank above the limit, 2 = rank above an extent (A_n^T A_n is singular)
  const int limit = N == 3 ? narrow_rank_bound(false) : CC_MAX_RANK_4;
  std::vector<int32_t> status(M, 0);
  for (int m = 0; m < M; m++) {
    const int R = c->hmodels[m].rank;
    if (R > limit)
      status[m] = 1;
    else
      for (int n = 0; n < N; n++)
        if (R > dims[n])
          status[m] = 2;
    if (status[m] == 0 && R > c->buffer_cols)
      return fail(c, "model %d has rank %d > buffer_size %d", m, R, c->buffer_cols);
  }

  // batches, and every model's jobs in the contraction steps s = 1 .. N-1 (output of step s: chain[(s - 1) & 1])
  long long rest = 1; // prod_{n >= 2} I_n
  for (int n = 2; n < N; n++)
    rest *= dims[n];
  const long long ldT = (long long)dims[1] * rest;
  auto out_size = [&](int R, int step) { // (prod_{n > step} I_n) * R^(step + 1)
    long long v = 1;
    for (int n = step + 1; n < N; n++)
      v *= dims[n];
    for (int k = 0; k <= step; k++)
      v *= R;
    return v;
  };
  const long long cap = (long long)(CC_BATCH_CAP_BYTES / 8);
  std::vector<CcModel> bm;
  std::vector<int> bstart{0};       // batch b: bm[bstart[b] .. bstart[b + 1])
  std::vector<int> bcols;
  std::vector<long long> bchain[2];
  int cols = 0, max_cols = 0;
  long long ch[2] = {0, 0}, max_chain[2] = {0, 0};
  auto close_batch = [&]() {
    bstart.push_back((int)bm.size());
    bcols.push_back(cols);
    max_cols = std::max(max_cols, cols);
    for (int k = 0; k < 2; k++) {
      bchain[k].push_back(ch[k]);
      max_chain[k] = std::max(max_chain[k], ch[k]);
      ch[k] = 0;
    }
    cols = 0;
  };
  for (int m = 0; m < M; m++) {
    if (status[m] != 0)
      continue;
    const HostModel &hm = c->hmodels[m];
    const int R = hm.rank;
    long long add[2] = {0, 0};
    for (int st = 1; st < N; st++)
      add[(st - 1) & 1] = std::max(add[(st - 1) & 1], out_size(R, st));
    const bool full = cols + R > c->buffer_cols || (long long)(cols + R) * ldT > cap || ch[0] + add[0] > cap ||
                      ch[1] + add[1] > cap;
    if (cols > 0 && full)
      close_batch();
    bm.push_back(CcModel{m, R, hm.home_col, cols, hm.jk_mode == 0 ? hm.jk_fiber : -1});
    cols += R;
    ch[0] += add[0];
    ch[1] += add[1];
  }
  if (cols > 0)
    close_batch();
  const int n_batches = (int)bcols.size(), n_bm = (int)bm.size();
  // jobs[(step - 1) * n_bm + i] for batch model i; offsets and first tiles count from the start of its batch
  std::vector<CcJob> jobs((size_t)(N - 1) * n_bm);
  std::vector<long long> tiles((size_t)(N - 1) * n_batches, 0);
  for (int b = 0; b < n_batches; b++)
    for (int st = 1; st < N; st++) {
      long long off = 0, t0 = 0;
      for (int i = bstart[b]; i < bstart[b + 1]; i++) {
        CcJob &j = jobs[(size_t)(st - 1) * n_bm + i];
        const int R = bm[i].rank;
        j.R = R;
        j.bcol = bm[i].bcol;
        j.in_off = st == 1 ? (long long)bm[i].bcol * ldT : jobs[(size_t)(st - 2) * n_bm + i].out_off;
        j.out_off = off;
        j.M = out_size(R, st) / R;
        j.tile0 = t0;
        off += out_size(R, st);
        t0 += (j.M + CC_CHAIN_MT - 1) / CC_CHAIN_MT;
      }
      tiles[(size_t)(st - 1) * n_batches + b] = t0;
    }

  // workspace: grown when this call needs more than the last one; 2 GB of device memory stay free
  const size_t job_bytes = jobs.size() * sizeof(CcJob), table_bytes = job_bytes + bm.size() * sizeof(CcModel);
  {
    size_t need = 0;
    auto more = [&](size_t cap_now, size_t n, size_t elem) { need += cap_now >= n ? 0 : n * elem; };
    for (int n = 0; n < N; n++) {
      if (!c->fitted)
        more(w.cap_F[n], (size_t)geo.ldF[n] * c->queued_cols, 8);
      more(w.cap_P[n], (size_t)geo.ldF[n] * max_cols, 8);
    }
    more(w.cap_T, (size_t)ldT * max_cols, 8);
    more(w.cap_chain, (size_t)std::max(max_chain[0], max_chain[1]), 16);
    size_t free_b = 0, total_b = 0;
    CU_TRY(c, cudaMemGetInfo(&free_b, &total_b));
    if (need + CC_HEADROOM_BYTES > free_b)
      return fail(c, "core consistency needs %.1f GB more device memory, %.1f GB are free", need / 1e9, free_b / 1e9);
  }
  const double *F[CALS_MAX_MODES] = {};
  const double *lambda = nullptr;
  for (int n = 0; n < N; n++) {
    if (c->fitted) { // after run / rerun: the fitted factors and lambda
      F[n] = c->bufs.fac.home[n];
      lambda = c->d_lambda;
    } else { // the queue as enqueued, lambda = 1 (the pinned staging already has the device layout)
      const size_t count = (size_t)geo.ldF[n] * c->queued_cols;
      if (cc_grow(c, &w.F[n], &w.cap_F[n], count))
        return 1;
      CU_TRY(c, cudaMemcpyAsync(w.F[n], c->h_in[n], count * 8, cudaMemcpyHostToDevice, s));
      F[n] = w.F[n];
    }
    if (cc_grow(c, &w.P[n], &w.cap_P[n], (size_t)geo.ldF[n] * max_cols))
      return 1;
  }
  if (cc_grow(c, &w.T, &w.cap_T, (size_t)ldT * max_cols))
    return 1;
  if (w.cap_chain < (size_t)std::max(max_chain[0], max_chain[1])) {
    size_t dummy = 0;
    if (cc_grow(c, &w.chain[0], &w.cap_chain, (size_t)std::max(max_chain[0], max_chain[1])) ||
        cc_grow(c, &w.chain[1], &dummy, w.cap_chain))
      return 1;
  }
  unsigned char *tab = nullptr;
  if (cc_grow(c, (unsigned char **)&w.tables, &w.cap_tables, table_bytes) ||
      cc_grow(c, &w.st, &w.cap_st, (size_t)std::max(n_batches, 1)) || cc_grow(c, &w.cc, &w.cap_models, (size_t)M))
    return 1;
  if (w.cap_models > 0) {
    size_t cs = 0, cf = 0;
    if (cc_grow(c, &w.status, &cs, w.cap_models) || cc_grow(c, &w.fail, &cf, w.cap_models * N))
      return 1;
  }
  tab = (unsigned char *)w.tables;
  const CcJob *d_jobs = (const CcJob *)tab;
  const CcModel *d_bm = (const CcModel *)(tab + job_bytes);
  if (n_bm > 0) {
    std::vector<unsigned char> host(table_bytes);
    memcpy(host.data(), jobs.data(), job_bytes);
    memcpy(host.data() + job_bytes, bm.data(), bm.size() * sizeof(CcModel));
    CU_TRY(c, cudaMemcpyAsync(tab, host.data(), table_bytes, cudaMemcpyHostToDevice, s));
    std::vector<SchedState> sts(n_batches);
    for (int b = 0; b < n_batches; b++) {
      sts[b] = SchedState{};
      sts[b].C = sts[b].C_main = bcols[b];
    }
    CU_TRY(c, cudaMemcpyAsync(w.st, sts.data(), sts.size() * sizeof(SchedState), cudaMemcpyHostToDevice, s));
  }

  int max_dim = 0;
  for (int n = 0; n < N; n++)
    max_dim = std::max(max_dim, dims[n]);
  for (int b = 0; b < n_batches; b++) {
    const int i0 = bstart[b], nb = bstart[b + 1] - i0, C = bcols[b];
    // 1. pseudo-inverses
    CcPinvParams pp{};
    pp.n_modes = N;
    for (int n = 0; n < N; n++) {
      pp.dims[n] = dims[n];
      pp.ld[n] = geo.ldF[n];
      pp.F[n] = F[n];
      pp.P[n] = w.P[n];
    }
    pp.lambda = lambda;
    pp.models = d_bm + i0;
    pp.fail = w.fail;
    size_t smem = 0;
    for (int i = i0; i < i0 + nb; i++)
      smem = std::max(smem, cc_pinv_smem(bm[i].rank, cc_chunk_rows(bm[i].rank, max_dim) + 4));
    pp.max_rows = max_dim;
    if (raise_smem_limit(c, (const void *)corcon_pinv_kernel, smem))
      return 1;
    corcon_pinv_kernel<<<dim3(nb, N), CC_THREADS, smem, s>>>(pp);
    CU_TRY(c, cudaGetLastError());
    // 2. T = X x_0 P_0 over the batch's columns: pair_gemm_kernel on the 3-D view (I_0, I_1, prod_{n>=2} I_n) of Xp
    PairMaps maps{};
    PairGeom pg{};
    pg.E1 = dims[1];
    pg.E2 = (int)rest;
    pg.R = (int)ldT;
    pg.ldT = ldT;
    pg.Ip = dims[0];
    pg.mode_fast = 1;
    pg.mode_slow = 2;
    for (int n = 0; n < N; n++)
      pg.ldF[n] = geo.ldF[n];
    pg.ld_fast = geo.ldF[1];
    const int wm = pick_pair_wm(pg.E1, pg.E2, C, c->sm_count);
    {
      cuuint64_t dx[3] = {(cuuint64_t)dims[0], (cuuint64_t)dims[1], (cuuint64_t)rest};
      cuuint64_t sx[2] = {(cuuint64_t)c->ldX0 * 8, (cuuint64_t)c->ldX0 * dims[1] * 8};
      cuuint32_t bx[3] = {(cuuint32_t)KT, 8, (cuuint32_t)wm};
      cuuint64_t d2[2] = {(cuuint64_t)dims[0], (cuuint64_t)C};
      cuuint64_t s2[1] = {(cuuint64_t)geo.ldF[0] * 8};
      cuuint32_t b2[2] = {(cuuint32_t)KT, (cuuint32_t)TILE_N};
      if (encode_map(c, &maps.X, c->Xp, 3, dx, sx, bx) || encode_map(c, &maps.B[0], w.P[0], 2, d2, s2, b2))
        return 1;
      maps.B[1] = maps.B[0];
    }
    const SchedState *st = w.st + b;
    int rc;
    switch (wm) {
    case 4:
      rc = launch_cc_pair_gemm<4>(c, maps, pg, st, w.T);
      break;
    case 5:
      rc = launch_cc_pair_gemm<5>(c, maps, pg, st, w.T);
      break;
    case 6:
      rc = launch_cc_pair_gemm<6>(c, maps, pg, st, w.T);
      break;
    case 7:
      rc = launch_cc_pair_gemm<7>(c, maps, pg, st, w.T);
      break;
    default:
      rc = launch_cc_pair_gemm<8>(c, maps, pg, st, w.T);
    }
    if (rc)
      return 1;
    // 3. the per-model chain, one launch per contracted mode
    for (int stp = 1; stp < N; stp++) {
      const long long grid = tiles[(size_t)(stp - 1) * n_batches + b];
      if (grid > 0x7fffffffLL)
        return fail(c, "core consistency: %lld tiles in one contraction step", grid);
      const double *in = stp == 1 ? w.T : w.chain[(stp - 2) & 1];
      corcon_chain_kernel<<<(unsigned)grid, CC_THREADS, 0, s>>>(d_jobs + (size_t)(stp - 1) * n_bm + i0, nb, dims[stp],
                                                                 in, w.P[stp], geo.ldF[stp], w.chain[(stp - 1) & 1]);
      CU_TRY(c, cudaGetLastError());
    }
    corcon_final_kernel<<<nb, CC_FINAL_THREADS, 0, s>>>(d_bm + i0, d_jobs + (size_t)(N - 2) * n_bm + i0, N,
                                                        w.chain[(N - 2) & 1], w.fail, w.cc, w.status);
    CU_TRY(c, cudaGetLastError());
  }

  std::vector<double> dcc(M);
  std::vector<int32_t> dst(M);
  if (n_bm > 0) {
    CU_TRY(c, cudaMemcpyAsync(dcc.data(), w.cc, (size_t)M * 8, cudaMemcpyDeviceToHost, s));
    CU_TRY(c, cudaMemcpyAsync(dst.data(), w.status, (size_t)M * 4, cudaMemcpyDeviceToHost, s));
  }
  CU_TRY(c, cudaStreamSynchronize(s));
  for (const CcModel &x : bm)
    status[x.model] = dst[x.model];
  for (int m = 0; m < M; m++) {
    cc_out[m] = status[m] == 0 ? dcc[m] : std::numeric_limits<double>::quiet_NaN();
    if (status_out)
      status_out[m] = status[m];
  }
  return 0;
}

} // namespace

// =================================================================================================================
extern "C" {

const char *cals_b200_version(void) { return "cals_b200 0.1 (sm_100a)"; }

const char *cals_b200_last_error(const cals_b200_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int cals_b200_create(cals_b200_ctx **out, int device) {
  if (!out)
    return fail(nullptr, "null ctx pointer");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, "no CUDA device available (%s): the B200 path has no CPU fallback",
                e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  if (device < 0 || device >= ndev)
    return fail(nullptr, "device %d out of range (have %d)", device, ndev);
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess)
    return fail(nullptr, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, "device %d is sm_%d%d; this library contains sm_100a code only", device, prop.major,
                prop.minor);
  cals_b200_ctx *c = new cals_b200_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaStreamCreate(&c->stream)) != cudaSuccess) {
    fail(nullptr, "cudaSetDevice/cudaStreamCreate: %s", cudaGetErrorString(e));
    delete c;
    return 1;
  }
  void *fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
    fail(nullptr, "cuTensorMapEncodeTiled not available from the driver");
    delete c;
    return 1;
  }
  c->encode = (PFN_encodeTiled)fn;
  bool aux_ok = cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking) == cudaSuccess;
  for (int n = 0; n < CALS_MAX_MODES && aux_ok; n++)
    aux_ok = cudaEventCreateWithFlags(&c->ev_fork[n], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&c->ev_join[n], cudaEventDisableTiming) == cudaSuccess;
  if (!aux_ok) {
    fail(nullptr, "cannot create the auxiliary stream / events");
    delete c;
    return 1;
  }
  if (cudaHostAlloc((void **)&c->h_flags, 64, cudaHostAllocMapped) != cudaSuccess ||
      cudaHostGetDevicePointer((void **)&c->d_flags, c->h_flags, 0) != cudaSuccess) {
    fail(nullptr, "cannot allocate mapped host flags");
    delete c;
    return 1;
  }
  memset(c->h_flags, 0, 64);
  *out = c;
  return 0;
}

int cals_b200_destroy(cals_b200_ctx *c) {
  if (!c)
    return 0;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  release_tensor(c);
  drop_iteration_graph(c);
  if (c->d_st)
    cudaFree(c->d_st);
  if (c->d_iter_cols)
    cudaFree(c->d_iter_cols);
  release_comm(c);
  if (c->h_flags)
    cudaFreeHost(c->h_flags);
  for (auto &p : c->h_home)
    if (p)
      cudaFreeHost(p);
  for (auto &p : c->h_in)
    if (p)
      cudaFreeHost(p);
  if (c->h_norm)
    cudaFreeHost(c->h_norm);
  if (c->h_lambda)
    cudaFreeHost(c->h_lambda);
  if (c->h_desc_pin)
    cudaFreeHost(c->h_desc_pin);
  if (c->norm_partial)
    cudaFree(c->norm_partial);
  if (c->x_stage)
    cudaFree(c->x_stage);
  for (auto e : c->ev_pool)
    cudaEventDestroy(e);
  for (int n = 0; n < CALS_MAX_MODES; n++) {
    if (c->ev_fork[n])
      cudaEventDestroy(c->ev_fork[n]);
    if (c->ev_join[n])
      cudaEventDestroy(c->ev_join[n]);
  }
  if (c->stream2)
    cudaStreamDestroy(c->stream2);
  cudaStreamDestroy(c->stream);
  delete c;
  return 0;
}

int cals_b200_set_tensor(cals_b200_ctx *c, int n_modes, const uint64_t *modes, const double *host_X) {
  if (!c || !modes || !host_X)
    return fail(c, "null argument");
  cudaSetDevice(c->device);
  return install_tensor(c, n_modes, modes, host_X, false);
}

int cals_b200_set_tensor_dev(cals_b200_ctx *c, int n_modes, const uint64_t *modes, const double *X_dev) {
  if (!c || !modes || !X_dev)
    return fail(c, "null argument");
  cudaSetDevice(c->device);
  return install_tensor(c, n_modes, modes, X_dev, true);
}

int cals_b200_set_tensor_slab(cals_b200_ctx *c, int n_modes, const uint64_t *modes, int slice_mode,
                              const uint64_t *cuts, const double *host_slab) {
  if (!c || !modes || !cuts || !host_slab)
    return fail(c, "null argument");
  cudaSetDevice(c->device);
  if (slice_mode < 0 || slice_mode >= n_modes)
    return fail(c, "slice_mode %d out of range", slice_mode);
  const int W = c->comm_world;
  if (cuts[0] != 0 || cuts[W] != modes[slice_mode])
    return fail(c, "slab boundaries must run from 0 to the extent of mode %d", slice_mode);
  for (int r = 0; r < W; r++)
    if (cuts[r + 1] <= cuts[r] || (cuts[r] & 1))
      return fail(c, "slab %d is empty or starts at an odd row", r);
  for (int r = 0; r <= W; r++)
    c->cuts[r] = (int)cuts[r];
  return install_tensor(c, n_modes, modes, host_slab, false, slice_mode, (long long)cuts[c->comm_rank],
                        (long long)cuts[c->comm_rank + 1]);
}

int cals_b200_set_tensor_norm(cals_b200_ctx *c, double norm) {
  if (!c)
    return 1;
  if (!c->have_tensor)
    return fail(c, "no tensor set");
  if (!(norm > 0.0))
    return fail(c, "the tensor norm must be positive");
  c->x_norm = norm;
  c->x_norm_valid = true;
  c->x_norm_override = true;
  return 0;
}

int cals_b200_comm_alloc(cals_b200_ctx *c, int rank, int world, uint64_t capacity_doubles, void *ipc_handle_out) {
  if (!c)
    return 1;
  if (world < 1 || world > CALS_MAX_PEERS || rank < 0 || rank >= world)
    return fail(c, "rank %d / world %d out of range (at most %d GPUs)", rank, world, CALS_MAX_PEERS);
  cudaSetDevice(c->device);
  CU_TRY(c, cudaStreamSynchronize(c->stream));
  release_comm(c);
  c->comm_rank = rank;
  c->comm_world = world;
  const size_t bytes = COMM_FLAG_BYTES + 2 * (size_t)capacity_doubles * 8;
  CU_TRY(c, cudaMalloc(&c->xblock, bytes));
  CU_TRY(c, cudaMemset(c->xblock, 0, bytes));
  c->xcap = (size_t)capacity_doubles;
  c->seq_base = 0;
  c->peer_block[rank] = c->xblock;
  if (ipc_handle_out) {
    cudaIpcMemHandle_t h;
    CU_TRY(c, cudaIpcGetMemHandle(&h, c->xblock));
    static_assert(sizeof(h) == 64, "cals_b200.h documents 64-byte handles");
    memcpy(ipc_handle_out, &h, sizeof h);
  }
  c->comm_connected = (world == 1);
  return 0;
}

int cals_b200_comm_local_block(cals_b200_ctx *c, void **block_dev_out) {
  if (!c || !block_dev_out)
    return fail(c, "null argument");
  if (!c->xblock)
    return fail(c, "cals_b200_comm_alloc has not been called");
  *block_dev_out = c->xblock;
  return 0;
}

int cals_b200_comm_connect(cals_b200_ctx *c, const void *ipc_handles, void *const *peer_blocks_dev,
                           const int *peer_devices) {
  if (!c)
    return 1;
  if (!c->xblock)
    return fail(c, "cals_b200_comm_alloc has not been called");
  if (!ipc_handles && !(peer_blocks_dev && peer_devices))
    return fail(c, "pass either the IPC handles of all ranks or their device pointers and device ordinals");
  cudaSetDevice(c->device);
  for (int r = 0; r < c->comm_world; r++) {
    if (r == c->comm_rank)
      continue;
    if (ipc_handles) { // one process per GPU
      cudaIpcMemHandle_t h;
      memcpy(&h, (const char *)ipc_handles + (size_t)r * sizeof h, sizeof h);
      void *p = nullptr;
      CU_TRY(c, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
      c->peer_block[r] = p;
      c->peer_is_ipc[r] = true;
    } else { // several GPUs driven by one process
      int can = 0;
      CU_TRY(c, cudaDeviceCanAccessPeer(&can, c->device, peer_devices[r]));
      if (!can)
        return fail(c, "device %d cannot access device %d", c->device, peer_devices[r]);
      cudaError_t e = cudaDeviceEnablePeerAccess(peer_devices[r], 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled)
        cudaGetLastError();
      else if (e != cudaSuccess)
        return fail(c, "cudaDeviceEnablePeerAccess(%d): %s", peer_devices[r], cudaGetErrorString(e));
      c->peer_block[r] = peer_blocks_dev[r];
      c->peer_is_ipc[r] = false;
    }
  }
  c->comm_connected = true;
  return 0;
}

int cals_b200_comm_disconnect(cals_b200_ctx *c) {
  if (!c)
    return 1;
  cudaSetDevice(c->device);
  CU_TRY(c, cudaStreamSynchronize(c->stream));
  disconnect_peers(c);
  if (c->xblock)
    c->peer_block[c->comm_rank] = c->xblock;
  return 0;
}

int cals_b200_configure(cals_b200_ctx *c, uint64_t buffer_cols, uint64_t max_iterations, double tol, unsigned flags) {
  if (!c)
    return 1;
  if (buffer_cols < 1 || buffer_cols > (1u << 24))
    return fail(c, "buffer_cols out of range");
  if (max_iterations < 1 || max_iterations > 0x7fffffffull)
    return fail(c, "max_iterations out of range");
  if ((int)buffer_cols != c->buffer_cols)
    c->uploaded = false;
  c->buffer_cols = (int)buffer_cols;
  c->max_iter = (int)max_iterations;
  c->tol = tol;
  c->flags = flags;
  return 0;
}

int cals_b200_set_line_search(cals_b200_ctx *c, int enabled, int method, int interval, double step) {
  if (!c)
    return 1;
  if (enabled) {
    if (method != 0 && method != 1)
      return fail(c, "line search method %d is not available (0 = no error checking, 1 = error checking, serial)",
                  method);
    if (interval < 2)
      return fail(c, "line search interval must be at least 2");
  }
  if ((enabled != 0) != (c->ls_enabled != 0) || method != c->ls_method)
    c->uploaded = false;
  c->ls_enabled = enabled ? 1 : 0;
  c->ls_method = method;
  c->ls_interval = interval;
  c->ls_step = step;
  return 0;
}

int cals_b200_line_search_counts(cals_b200_ctx *c, uint64_t *performed, uint64_t *failed) {
  if (!c)
    return 1;
  if (performed)
    *performed = c->last_ls_performed;
  if (failed)
    *failed = c->last_ls_failed;
  return 0;
}

int cals_b200_set_timing(cals_b200_ctx *c, int level) {
  if (!c)
    return 1;
  c->timing = level;
  return 0;
}

int cals_b200_set_mttkrp_variant(cals_b200_ctx *c, int variant) {
  if (!c)
    return 1;
  if (variant != CALS_B200_MTTKRP_DMMA && variant != CALS_B200_MTTKRP_NAIVE)
    return fail(c, "unknown MTTKRP variant %d", variant);
  c->variant = variant;
  return 0;
}

int cals_b200_set_pair_node(cals_b200_ctx *c, int enabled) {
  if (!c)
    return 1;
  c->pair_node = enabled ? 1 : 0;
  return 0;
}

// Pinned input staging of mode n for at least `cols` queued columns; what is already queued is kept.
static int reserve_input_staging(cals_b200_ctx *c, int n, size_t cols, bool geometric) {
  const size_t ld = (size_t)c->geo.ldF[n];
  const size_t need = ld * cols;
  if (need <= c->h_in_cap[n])
    return 0;
  const size_t cap = geometric ? std::max(need, std::max<size_t>(2 * c->h_in_cap[n], ld * 256)) : need;
  double *fresh = nullptr;
  CU_TRY(c, cudaHostAlloc((void **)&fresh, cap * 8, cudaHostAllocDefault));
  if (c->h_in[n]) {
    CU_TRY(c, cudaStreamSynchronize(c->stream)); // an upload from the old block may still be in flight
    memcpy(fresh, c->h_in[n], ld * c->queued_cols * 8);
    cudaFreeHost(c->h_in[n]);
  }
  c->h_in[n] = fresh;
  c->h_in_cap[n] = cap;
  return 0;
}

int cals_b200_clear_models(cals_b200_ctx *c) {
  if (!c)
    return 1;
  c->hmodels.clear();
  c->hdesc.clear();
  c->h_active.clear();
  c->queued_cols = 0;
  c->uploaded = false;
  c->fitted = false;
  c->results_fresh = false;
  return 0;
}

// validation shared by the two enqueue entry points; on success fills `hm` (home_col = first free staging column)
static int check_model(cals_b200_ctx *c, uint64_t rank, const double *const *host_factors, int jk_mode, int64_t jk_fiber,
                       int home_col, int id, HostModel *hm) {
  if (rank < 1 || rank > 4096)
    return fail(c, "rank %llu out of range", (unsigned long long)rank);
  if (check_nnls_rank(c, id, (int)rank))
    return 1;
  const Geom &geo = c->geo;
  if (jk_mode >= geo.n_modes)
    return fail(c, "jk_mode %d out of range", jk_mode);
  // Leave-one-out norms exist for mode 0 only, as in the reference (utils::calculate_jackknifing_norms,
  // src/utils/utils.cpp:103-152; generate_jk_ktensors flags mode 0, :40-51): another mode would index that table with
  // a fibre of the wrong mode and silently give a wrong error / fit / eviction decision.
  if (jk_mode > 0)
    return fail(c, "jackknife models must leave out a sample of mode 0 (jk_mode %d): the leave-one-out norms "
                   "||X||_jk are kept for mode 0 only, as in the reference", jk_mode);
  if (jk_mode >= 0 && (jk_fiber < 0 || jk_fiber >= geo.dims[jk_mode]))
    return fail(c, "jk_fiber %lld out of range", (long long)jk_fiber);
  if (jk_mode >= 0 && c->slice_mode >= 0)
    return fail(c, "jackknife models are not supported on a sliced tensor (shard the sub-models instead)");
  for (int n = 0; n < geo.n_modes; n++)
    if (!host_factors[n])
      return fail(c, "factor %d is null", n);
  hm->rank = (int)rank;
  hm->jk_mode = jk_mode < 0 ? -1 : jk_mode;
  hm->jk_fiber = jk_mode < 0 ? 0 : (int)jk_fiber;
  hm->home_col = home_col;
  return 0;
}

// copy one model's factors into the pinned input staging at its home columns (pitch ldF, pad row zeroed)
static void stage_model(cals_b200_ctx *c, const HostModel &hm, const double *const *host_factors) {
  const Geom &geo = c->geo;
  for (int n = 0; n < geo.n_modes; n++) {
    const int rows = geo.dims[n], ld = geo.ldF[n];
    double *dst = c->h_in[n] + (size_t)ld * hm.home_col;
    if (ld == rows)
      memcpy(dst, host_factors[n], (size_t)rows * hm.rank * 8);
    else
      for (int j = 0; j < hm.rank; j++) {
        memcpy(dst + (size_t)j * ld, host_factors[n] + (size_t)j * rows, (size_t)rows * 8);
        dst[(size_t)j * ld + rows] = 0.0;
      }
  }
}

int cals_b200_enqueue_model(cals_b200_ctx *c, uint64_t rank, const double *const *host_factors, int jk_mode,
                            int64_t jk_fiber, int *model_id) {
  if (!c || !host_factors)
    return fail(c, "null argument");
  if (!c->have_tensor)
    return fail(c, "set the tensor before enqueueing models");
  HostModel hm;
  if (check_model(c, rank, host_factors, jk_mode, jk_fiber, c->queued_cols, (int)c->hmodels.size(), &hm))
    return 1;
  for (int n = 0; n < c->geo.n_modes; n++)
    if (reserve_input_staging(c, n, (size_t)c->queued_cols + rank, true))
      return 1;
  stage_model(c, hm, host_factors);
  c->queued_cols += (int)rank;
  c->hmodels.push_back(hm);
  c->uploaded = false;
  c->fitted = false;
  if (model_id)
    *model_id = (int)c->hmodels.size() - 1;
  return 0;
}

int cals_b200_enqueue_models(cals_b200_ctx *c, uint64_t n_models, const uint64_t *ranks,
                             const double *const *host_factors, const int *jk_modes, const int64_t *jk_fibers) {
  if (!c || !ranks || !host_factors)
    return fail(c, "null argument");
  if (!c->have_tensor)
    return fail(c, "set the tensor before enqueueing models");
  const int N = c->geo.n_modes;
  // validate everything first: a rejected model leaves the queue as it was
  std::vector<HostModel> fresh((size_t)n_models);
  int col = c->queued_cols;
  size_t rows_sum = 0;
  for (int n = 0; n < N; n++)
    rows_sum += (size_t)c->geo.dims[n];
  for (uint64_t m = 0; m < n_models; m++) {
    if (check_model(c, ranks[m], host_factors + m * N, jk_modes ? jk_modes[m] : -1, jk_fibers ? jk_fibers[m] : 0, col,
                    (int)(c->hmodels.size() + m), &fresh[m]))
      return 1;
    col += (int)ranks[m];
  }
  for (int n = 0; n < N; n++) // one pinned allocation per mode for the whole queue
    if (reserve_input_staging(c, n, (size_t)col, false))
      return 1;
  parallel_models((size_t)n_models, rows_sum * (size_t)(col - c->queued_cols) * 8, [&](size_t lo, size_t hi) {
    for (size_t m = lo; m < hi; m++)
      stage_model(c, fresh[m], host_factors + m * N);
  });
  c->queued_cols = col;
  c->hmodels.insert(c->hmodels.end(), fresh.begin(), fresh.end());
  c->uploaded = false;
  c->fitted = false;
  return 0;
}

int cals_b200_run(cals_b200_ctx *c, cals_b200_report *rep) {
  if (!c)
    return 1;
  cudaSetDevice(c->device);
  static const bool trace = getenv("CALS_B200_TRACE") != nullptr; // host-side phase times on stderr
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
  const auto t0 = now();
  if (prepare_run(c))
    return 1;
  const auto t1 = now();
  if (run_loop(c, rep, false))
    return 1;
  const auto t2 = now();
  const int rc = download_results(c);
  if (trace)
    fprintf(stderr, "[cals_b200] run: prepare %.3f ms, loop %.3f ms (device %.3f ms), download %.3f ms\n", ms(t0, t1),
            ms(t1, t2), rep ? rep->device_ms : 0.0, ms(t2, now()));
  return rc;
}

int cals_b200_rerun(cals_b200_ctx *c, cals_b200_report *rep) {
  if (!c)
    return 1;
  cudaSetDevice(c->device);
  if (!c->uploaded)
    return fail(c, "rerun needs a previous cals_b200_run with the same queue and buffer size");
  return run_loop(c, rep, true);
}

int cals_b200_fetch_model(cals_b200_ctx *c, int model_id, double *const *factors_out, double *lambda_out,
                          cals_b200_model_stats *stats) {
  if (!c)
    return 1;
  cudaSetDevice(c->device);
  if (model_id < 0 || model_id >= (int)c->hdesc.size())
    return fail(c, "model id %d out of range", model_id);
  if (download_results(c))
    return 1;
  copy_model_out(c, model_id, factors_out, lambda_out, stats);
  return 0;
}

int cals_b200_fetch_all(cals_b200_ctx *c, double *const *factors_out, double *const *lambda_out,
                        cals_b200_model_stats *stats) {
  if (!c)
    return 1;
  cudaSetDevice(c->device);
  if (download_results(c))
    return 1;
  const int N = c->geo.n_modes;
  size_t rows_sum = 0;
  for (int n = 0; n < N; n++)
    rows_sum += (size_t)c->geo.dims[n];
  parallel_models(c->hdesc.size(), factors_out ? rows_sum * (size_t)c->total_cols * 8 : 0, [&](size_t lo, size_t hi) {
    for (size_t m = lo; m < hi; m++)
      copy_model_out(c, (int)m, factors_out ? factors_out + m * N : nullptr, lambda_out ? lambda_out[m] : nullptr,
                     stats ? stats + m : nullptr);
  });
  return 0;
}

// Layout shared by both calls: active[n] -> I_n x rank bytes, row-major (byte [row * rank + col]), 1 = constrained.
static long long model_act_offset(cals_b200_ctx *c, int model_id, long long *sum_rows_out) {
  long long sum_rows = 0, off = 0;
  for (int n = 0; n < c->geo.n_modes; n++)
    sum_rows += c->geo.dims[n];
  for (int m = 0; m < model_id; m++)
    off += sum_rows * c->hmodels[m].rank;
  *sum_rows_out = sum_rows;
  return off;
}

int cals_b200_set_model_active_set(cals_b200_ctx *c, int model_id, const uint8_t *const *active) {
  if (!c || !active)
    return fail(c, "null argument");
  if (model_id < 0 || model_id >= (int)c->hmodels.size())
    return fail(c, "model id %d out of range", model_id);
  long long sum_rows = 0, total = 0;
  const long long off = model_act_offset(c, model_id, &sum_rows);
  for (auto &hm : c->hmodels)
    total += sum_rows * hm.rank;
  if ((long long)c->h_active.size() != total) { // models queued since the last sizing: extend with "all active"
    c->h_active.resize((size_t)total, 1);
  }
  long long o = off;
  for (int n = 0; n < c->geo.n_modes; n++) {
    const long long cnt = (long long)c->geo.dims[n] * c->hmodels[model_id].rank;
    if (!active[n])
      return fail(c, "active set of mode %d is null", n);
    memcpy(&c->h_active[(size_t)o], active[n], (size_t)cnt);
    o += cnt;
  }
  return 0;
}

int cals_b200_fetch_model_active_set(cals_b200_ctx *c, int model_id, uint8_t *const *active_out) {
  if (!c || !active_out)
    return fail(c, "null argument");
  if (model_id < 0 || model_id >= (int)c->hdesc.size() || !c->uploaded || !c->d_active)
    return fail(c, "no run to fetch the active set of model %d from", model_id);
  cudaSetDevice(c->device);
  long long sum_rows = 0;
  long long o = model_act_offset(c, model_id, &sum_rows);
  for (int n = 0; n < c->geo.n_modes; n++) {
    const long long cnt = (long long)c->geo.dims[n] * c->hmodels[model_id].rank;
    if (active_out[n])
      CU_TRY(c, cudaMemcpy(active_out[n], c->d_active + o, (size_t)cnt, cudaMemcpyDeviceToHost));
    o += cnt;
  }
  return 0;
}

int cals_b200_tensor_norm(cals_b200_ctx *c, double *norm_out) {
  if (!c || !norm_out)
    return fail(c, "null argument");
  if (!c->have_tensor)
    return fail(c, "no tensor set");
  cudaSetDevice(c->device);
  if (ensure_host_norm(c))
    return 1;
  *norm_out = c->x_norm;
  return 0;
}

int cals_b200_jk_norms(cals_b200_ctx *c, double *out) {
  if (!c || !out)
    return fail(c, "null argument");
  if (!c->have_tensor)
    return fail(c, "no tensor set");
  cudaSetDevice(c->device);
  CU_TRY(c, cudaMemcpy(out, c->jk_norms, (size_t)c->geo.dims[0] * 8, cudaMemcpyDeviceToHost));
  return 0;
}

int cals_b200_mttkrp(cals_b200_ctx *c, int mode, uint64_t cols, const double *const *host_factors, double *host_G,
                     int variant, int repeats, double *ms_out) {
  if (!c || !host_factors || !host_G)
    return fail(c, "null argument");
  if (!c->have_tensor)
    return fail(c, "no tensor set");
  cudaSetDevice(c->device);
  const Geom &geo = c->geo;
  if (mode < 0 || mode >= geo.n_modes)
    return fail(c, "mode out of range");
  if (cols < 1 || cols > (1u << 24))
    return fail(c, "cols out of range");
  if (ensure_dummy_state(c))
    return 1;
  Buffers b;
  int rc = alloc_buffers(c, b, (int)cols, false, 0);
  if (!rc) {
    for (int k = 0; k < geo.n_modes && !rc; k++) {
      if (k == mode)
        continue;
      if (!host_factors[k]) {
        rc = fail(c, "factor %d is null", k);
        break;
      }
      cudaError_t e = cudaMemcpy2DAsync(b.fac.buf[0][k], (size_t)geo.ldF[k] * 8, host_factors[k],
                                        (size_t)geo.dims[k] * 8, (size_t)geo.dims[k] * 8, cols,
                                        cudaMemcpyHostToDevice, c->stream);
      if (e != cudaSuccess)
        rc = fail(c, "upload of factor %d failed: %s", k, cudaGetErrorString(e));
    }
  }
  if (!rc) {
    cudaEvent_t e0 = get_event(c, 0), e1 = get_event(c, 1);
    if (repeats < 1)
      repeats = 1;
    if (c->slice_mode >= 0) // rows outside this device's slab are not produced: the hook returns them as zeros
      cudaMemsetAsync(b.G, 0, (size_t)geo.ldF[mode] * cols * 8, c->stream);
    c->pdl = false; // single launches in plain stream order
    mttkrp_plan_kernel<<<1, 32, 0, c->stream>>>(b.plans, (int)cols, b.narrow ? 1 : 0);
    rc = launch_mttkrp(c, b, mode, (int)cols, variant); // warm-up + result
    cudaEventRecord(e0, c->stream);
    for (int r = 1; r < repeats && !rc; r++)
      rc = launch_mttkrp(c, b, mode, (int)cols, variant);
    cudaEventRecord(e1, c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e == cudaSuccess)
      e = cudaGetLastError();
    if (e != cudaSuccess)
      rc = fail(c, "MTTKRP kernel failed: %s", cudaGetErrorString(e));
    if (!rc && ms_out) {
      float ms = 0;
      cudaEventElapsedTime(&ms, e0, e1);
      *ms_out = repeats > 1 ? ms / (repeats - 1) : 0.0;
    }
    if (!rc) {
      e = cudaMemcpy2D(host_G, (size_t)geo.dims[mode] * 8, b.G, (size_t)geo.ldF[mode] * 8,
                       (size_t)geo.dims[mode] * 8, cols, cudaMemcpyDeviceToHost);
      if (e != cudaSuccess)
        rc = fail(c, "download of G failed: %s", cudaGetErrorString(e));
    }
  }
  free_all(b.allocs);
  return rc;
}

int cals_b200_khatri_rao(cals_b200_ctx *c, const double *host_A, uint64_t rows_A, const double *host_B, uint64_t rows_B,
                         uint64_t cols, double *host_K) {
  if (!c || !host_A || !host_B || !host_K)
    return fail(c, "null argument");
  if (rows_A < 1 || rows_B < 1 || cols < 1 || rows_A > (1u << 30) || rows_B > (1u << 30) || cols > 65535 ||
      rows_A * rows_B > (1ull << 40))
    return fail(c, "khatri_rao: extents out of range (%llu x %llu rows, %llu columns)", (unsigned long long)rows_A,
                (unsigned long long)rows_B, (unsigned long long)cols);
  cudaSetDevice(c->device);
  const size_t nA = (size_t)rows_A * cols, nB = (size_t)rows_B * cols, nK = (size_t)rows_A * rows_B * cols;
  double *dA = nullptr, *dB = nullptr, *dK = nullptr;
  int rc = 0;
  cudaError_t e = cudaMalloc((void **)&dA, nA * 8);
  if (e == cudaSuccess)
    e = cudaMalloc((void **)&dB, nB * 8);
  if (e == cudaSuccess)
    e = cudaMalloc((void **)&dK, nK * 8);
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(dA, host_A, nA * 8, cudaMemcpyHostToDevice, c->stream);
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(dB, host_B, nB * 8, cudaMemcpyHostToDevice, c->stream);
  if (e == cudaSuccess) {
    const unsigned long long rows = rows_A * rows_B;
    dim3 grid((unsigned)((rows + 1023) / 1024), (unsigned)cols);
    khatri_rao_kernel<<<grid, 256, 0, c->stream>>>(dA, dB, (int)rows_A, (int)rows_B, dK);
    e = cudaMemcpyAsync(host_K, dK, nK * 8, cudaMemcpyDeviceToHost, c->stream);
  }
  if (e == cudaSuccess)
    e = cudaStreamSynchronize(c->stream);
  if (e == cudaSuccess)
    e = cudaGetLastError();
  if (e != cudaSuccess)
    rc = fail(c, "khatri_rao failed: %s", cudaGetErrorString(e));
  cudaFree(dA);
  cudaFree(dB);
  cudaFree(dK);
  return rc;
}

int cals_b200_fetch_iteration_cols(cals_b200_ctx *c, uint32_t *cols_out, uint64_t capacity, uint64_t *n_out) {
  if (!c || !n_out)
    return fail(c, "null argument");
  cudaSetDevice(c->device);
  const uint64_t logged = std::min<uint64_t>(c->last_global_iter, (uint64_t)ITER_LOG_CAP);
  *n_out = logged;
  const uint64_t n = std::min<uint64_t>(logged, capacity);
  if (n && cols_out) {
    if (!c->d_iter_cols)
      return fail(c, "no run to fetch the iteration log from");
    CU_TRY(c, cudaMemcpy(cols_out, c->d_iter_cols, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  }
  return 0;
}

void *cals_b200_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError(); // no device / out of pinned memory: the caller falls back to pageable memory
    return nullptr;
  }
  return p;
}

void cals_b200_host_free(void *p) {
  if (p)
    cudaFreeHost(p);
}

int cals_b200_stream(cals_b200_ctx *c, void **stream_out) {
  if (!c || !stream_out)
    return fail(c, "null argument");
  *stream_out = (void *)c->stream;
  return 0;
}

int cals_b200_device_info(cals_b200_ctx *c, int *sm_count, size_t *free_bytes, size_t *total_bytes) {
  if (!c)
    return 1;
  cudaSetDevice(c->device);
  if (sm_count)
    *sm_count = c->sm_count;
  size_t f = 0, t = 0;
  CU_TRY(c, cudaMemGetInfo(&f, &t));
  if (free_bytes)
    *free_bytes = f;
  if (total_bytes)
    *total_bytes = t;
  return 0;
}

int cals_b200_core_consistency(cals_b200_ctx *c, double *cc_out, int32_t *status_out) {
  if (!c || !cc_out)
    return fail(c, "null argument");
  cudaSetDevice(c->device);
  return core_consistency(c, cc_out, status_out);
}

} // extern "C"
