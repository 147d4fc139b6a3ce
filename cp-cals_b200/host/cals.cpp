// cals::cp_cals / cals::jk_cp_cals on the B200 (reference src/cals.cpp:19-446).
//
// What the reference does on the host inside its do/while loop -- admission, MTTKRP, per-model update, error, eviction,
// compaction -- runs on the device behind cals_b200_run (cp-cals_b200/csrc).  The host side left here is: validate the
// parameters, hand X and the queued models to the C ABI, copy the fitted models back into the caller's Ktensors and
// fill the report.  With CalsParams::devices = {d0, d1, ..} the model set is sharded over several GPUs of the box (X
// replicated, one host thread per device, no data-path collective).
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <map>
#include <memory>
#include <numeric>
#include <thread>

#include "cals.h"
#include "engine_pool.h"

namespace cals {
namespace detail {

namespace {
std::mutex g_pool_mu;
std::map<int, std::unique_ptr<EngineHandle>> g_pool;

struct PoolCleaner { // destroy the contexts before the CUDA runtime is torn down at exit
  ~PoolCleaner() {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    for (auto &kv : g_pool)
      if (kv.second->ctx)
        cals_b200_destroy(kv.second->ctx);
    g_pool.clear();
  }
} g_cleaner;
} // namespace

EngineHandle &engine_for_device(int device) {
  std::lock_guard<std::mutex> lk(g_pool_mu);
  auto it = g_pool.find(device);
  if (it != g_pool.end())
    return *it->second;
  auto h = std::make_unique<EngineHandle>();
  h->device = device;
  if (cals_b200_create(&h->ctx, device) != 0)
    throw B200Error(std::string("cals_b200_create(device ") + std::to_string(device) +
                    ") failed: " + cals_b200_last_error(nullptr));
  return *(g_pool[device] = std::move(h));
}

void check(EngineHandle &e, int rc, const char *what) {
  if (rc != 0)
    throw B200Error(std::string(what) + ": " + cals_b200_last_error(e.ctx));
}

// Content fingerprint: FNV-1a over the bit patterns of up to 4096 evenly spaced elements (plus the last one).  Writes
// through Tensor::get_data() / operator[] bypass the uid, so the skip below also asks for an unchanged sample; a caller
// who rewrites X in place between two calls and still sets cuda_no_tensor_alloc is caught unless every sampled element
// kept its value -- the reference trusts that flag blindly (src/als.cpp:146-152).
static uint64_t tensor_fingerprint(const Tensor &X) {
  const dim_t n = X.get_n_elements();
  const double *d = X.get_data();
  uint64_t h = 1469598103934665603ull;
  auto mix = [&h](double v) {
    uint64_t b;
    memcpy(&b, &v, 8);
    h = (h ^ b) * 1099511628211ull;
  };
  if (n == 0 || d == nullptr)
    return h;
  const dim_t step = std::max<dim_t>(1, n / 4096);
  for (dim_t i = 0; i < n; i += step)
    mix(d[i]);
  mix(d[n - 1]);
  return h ^ (uint64_t)n;
}

void upload_tensor(EngineHandle &e, const Tensor &X, bool may_skip) {
  const vector<dim_t> modes = X.get_modes();
  const uint64_t fp = tensor_fingerprint(X);
  if (may_skip && e.resident_data == X.get_data() && e.resident_modes == modes && e.resident_uid == X.get_uid() &&
      e.resident_fp == fp)
    return;
  std::vector<uint64_t> m(modes.begin(), modes.end());
  e.resident_data = nullptr;
  check(e, cals_b200_set_tensor(e.ctx, static_cast<int>(m.size()), m.data(), X.get_data()), "cals_b200_set_tensor");
  e.resident_data = X.get_data();
  e.resident_modes = modes;
  e.resident_uid = X.get_uid();
  e.resident_fp = fp;
}

RunResult run_on_device(int device, const Tensor &X, const std::vector<Ktensor *> &models, const RunOptions &opt) {
  static const bool trace = getenv("CALS_B200_TRACE") != nullptr; // host-side phase times on stderr
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
  const auto t_begin = now();
  EngineHandle &e = engine_for_device(device);
  std::lock_guard<std::mutex> lk(e.mu);
  RunResult out;
  if (models.empty())
    return out;
  const auto t_engine = now();
  upload_tensor(e, X, opt.skip_upload_if_resident);
  const auto t_upload = now();
  const unsigned flags = (opt.force_max_iter ? CALS_B200_FORCE_MAX_ITER : 0u) |
                         (opt.always_evict_first ? CALS_B200_ALWAYS_EVICT_FIRST : 0u) |
                         (opt.nnls ? CALS_B200_NNLS : 0u);
  // A buffer wider than the whole queue behaves exactly like one that just holds it (everything is admitted at once),
  // so the device buffers are sized by what can actually be resident.
  dim_t sum_ranks = 0;
  for (const Ktensor *kt : models)
    sum_ranks += kt->get_components();
  const dim_t buffer = std::max<dim_t>(std::min(opt.buffer_size, sum_ranks), 1);
  check(e, cals_b200_configure(e.ctx, buffer, opt.max_iterations, opt.tol, flags), "cals_b200_configure");
  check(e, cals_b200_set_line_search(e.ctx, opt.line_search, opt.ls_method, opt.ls_interval, opt.ls_step),
        "cals_b200_set_line_search");
  check(e, cals_b200_set_timing(e.ctx, opt.timing), "cals_b200_set_timing");
  check(e, cals_b200_set_pair_node(e.ctx, opt.pair_node), "cals_b200_set_pair_node");
  check(e, cals_b200_clear_models(e.ctx), "cals_b200_clear_models");

  const dim_t N = X.get_n_modes();
  {
    std::vector<const double *> in(models.size() * N);
    std::vector<uint64_t> ranks(models.size());
    std::vector<int> jk_modes(models.size());
    std::vector<int64_t> jk_fibers(models.size());
    for (size_t m = 0; m < models.size(); m++) {
      const Ktensor *kt = models[m];
      if (kt->get_n_modes() != N)
        throw B200Error("cp_cals: a Ktensor has a different number of modes than the tensor");
      for (dim_t n = 0; n < N; n++) {
        if (kt->get_factor(n).get_rows() != X.get_modes()[n])
          throw B200Error("cp_cals: a Ktensor factor does not match the tensor extents");
        in[m * N + n] = kt->get_factor(n).get_data();
      }
      ranks[m] = kt->get_components();
      jk_modes[m] = kt->is_jk() ? (int)kt->get_jk_mode() : -1;
      jk_fibers[m] = kt->is_jk() ? (int64_t)kt->get_jk_fiber() : 0;
    }
    check(e, cals_b200_enqueue_models(e.ctx, models.size(), ranks.data(), in.data(), jk_modes.data(), jk_fibers.data()),
          "cals_b200_enqueue_models");
  }
  if (opt.nnls) { // warm-start active sets live in the Ktensor (reference include/ktensor.h:36); fresh ones are all-true
    std::vector<std::vector<uint8_t>> bytes(N);
    std::vector<const uint8_t *> ptrs(N);
    for (size_t m = 0; m < models.size(); m++) {
      Ktensor *kt = models[m];
      bool fresh = true;
      for (dim_t n = 0; n < N && fresh; n++)
        for (const auto &row : kt->get_active_set(n))
          for (bool a : row)
            fresh = fresh && a;
      if (fresh)
        continue;
      for (dim_t n = 0; n < N; n++) {
        const auto &as = kt->get_active_set(n);
        bytes[n].assign(as.size() * kt->get_components(), 1);
        for (size_t r = 0; r < as.size(); r++)
          for (size_t c = 0; c < as[r].size(); c++)
            bytes[n][r * kt->get_components() + c] = as[r][c] ? 1 : 0;
        ptrs[n] = bytes[n].data();
      }
      check(e, cals_b200_set_model_active_set(e.ctx, (int)m, ptrs.data()), "cals_b200_set_model_active_set");
    }
  }
  const auto t_queued = now();
  check(e, cals_b200_run(e.ctx, &out.rep), "cals_b200_run");
  const auto t_ran = now();
  if (trace)
    fprintf(stderr, "[cals] device %d: engine %.3f ms, set_tensor %.3f ms, queue %zu models %.3f ms, run %.3f ms\n",
            device, ms(t_begin, t_engine), ms(t_engine, t_upload), models.size(), ms(t_upload, t_queued),
            ms(t_queued, t_ran));
  check(e, cals_b200_line_search_counts(e.ctx, &out.ls_performed, &out.ls_failed), "cals_b200_line_search_counts");

  // results straight into the callers' storage (Ktensor::detach of the reference, src/ktensor.cpp:127-135)
  const size_t M = models.size();
  std::vector<double *> fptr(M * N), lptr(M);
  std::vector<cals_b200_model_stats> stats(M);
  for (size_t m = 0; m < M; m++) {
    for (dim_t n = 0; n < N; n++)
      fptr[m * N + n] = models[m]->get_factor(n).get_data();
    lptr[m] = models[m]->get_lambda().data();
  }
  check(e, cals_b200_fetch_all(e.ctx, fptr.data(), lptr.data(), stats.data()), "cals_b200_fetch_all");
  for (size_t m = 0; m < M; m++) {
    models[m]->set_iters(static_cast<dim_t>(stats[m].iters));
    models[m]->set_approximation_error(stats[m].error);
    models[m]->set_fit(stats[m].fit, stats[m].old_fit);
  }
  if (opt.nnls) {
    std::vector<std::vector<uint8_t>> bytes(N);
    std::vector<uint8_t *> ptrs(N);
    for (size_t m = 0; m < M; m++) {
      Ktensor *kt = models[m];
      for (dim_t n = 0; n < N; n++) {
        bytes[n].resize(kt->get_factor(n).get_rows() * kt->get_components());
        ptrs[n] = bytes[n].data();
      }
      check(e, cals_b200_fetch_model_active_set(e.ctx, (int)m, ptrs.data()), "cals_b200_fetch_model_active_set");
      for (dim_t n = 0; n < N; n++) {
        auto &as = kt->get_active_set(n);
        for (size_t r = 0; r < as.size(); r++)
          for (size_t c = 0; c < as[r].size(); c++)
            as[r][c] = bytes[n][r * kt->get_components() + c] != 0;
      }
    }
  }
  uint64_t n_it = 0;
  check(e, cals_b200_fetch_iteration_cols(e.ctx, nullptr, 0, &n_it), "cals_b200_fetch_iteration_cols");
  std::vector<uint32_t> c32(n_it);
  if (n_it)
    check(e, cals_b200_fetch_iteration_cols(e.ctx, c32.data(), n_it, &n_it), "cals_b200_fetch_iteration_cols");
  out.cols.assign(c32.begin(), c32.end());
  return out;
}

std::vector<dim_t> shard_slabs(dim_t extent, size_t n_parts) {
  std::vector<dim_t> cuts{0};
  for (size_t p = 1; p < n_parts; p++) {
    dim_t c = static_cast<dim_t>(static_cast<double>(p) * extent / n_parts / 2.0 + 0.5) * 2; // even boundaries
    cuts.push_back(std::min(std::max(c, cuts.back()), extent));
  }
  cuts.push_back(extent);
  return cuts;
}

// Config 5: X sliced along `slice_mode` over the devices, all models on every device, one host thread per device.
// Every device ends with the same (bit-identical) results; device 0's are written into the callers' Ktensors.
static RunResult run_sliced(const std::vector<int> &devices, int slice_mode, const Tensor &X,
                            const std::vector<Ktensor *> &models, const RunOptions &opt) {
  const size_t W = devices.size();
  const vector<dim_t> modes = X.get_modes();
  const dim_t N = modes.size();
  if (slice_mode < 0 || static_cast<dim_t>(slice_mode) >= N)
    throw B200Error("cp_cals: slice_mode out of range");
  for (size_t a = 0; a < W; a++)
    for (size_t b = a + 1; b < W; b++)
      if (devices[a] == devices[b])
        throw B200Error("cp_cals: a sliced tensor needs distinct devices (ranks wait for each other on the GPU)");
  const std::vector<dim_t> cuts = shard_slabs(modes[slice_mode], W);
  for (size_t r = 0; r < W; r++)
    if (cuts[r + 1] <= cuts[r])
      throw B200Error("cp_cals: more devices than (pairs of) rows in the sliced mode");
  dim_t sum_ranks = 0;
  for (const Ktensor *kt : models) {
    if (kt->is_jk())
      throw B200Error("cp_cals: jackknife models are not supported on a sliced tensor");
    sum_ranks += kt->get_components();
  }
  const dim_t buffer = std::max<dim_t>(std::min(opt.buffer_size, sum_ranks), 1);
  dim_t max_ld = 0;
  for (dim_t m : modes)
    max_ld = std::max(max_ld, (m + 1) / 2 * 2);
  std::vector<uint64_t> m64(modes.begin(), modes.end()), c64(cuts.begin(), cuts.end());

  std::vector<EngineHandle *> eng(W);
  std::vector<std::unique_lock<std::mutex>> locks;
  for (size_t r = 0; r < W; r++) {
    eng[r] = &engine_for_device(devices[r]);
    locks.emplace_back(eng[r]->mu);
    eng[r]->resident_data = nullptr;
  }
  // exchange blocks + peer mapping (one process drives all GPUs: plain peer pointers)
  std::vector<void *> blocks(W);
  for (size_t r = 0; r < W; r++) {
    check(*eng[r], cals_b200_comm_alloc(eng[r]->ctx, (int)r, (int)W, max_ld * buffer, nullptr), "cals_b200_comm_alloc");
    check(*eng[r], cals_b200_comm_local_block(eng[r]->ctx, &blocks[r]), "cals_b200_comm_local_block");
  }
  for (size_t r = 0; r < W; r++)
    check(*eng[r], cals_b200_comm_connect(eng[r]->ctx, nullptr, blocks.data(), devices.data()),
          "cals_b200_comm_connect");

  // slabs: contiguous for the last mode, gathered otherwise
  dim_t below = 1, above = 1;
  for (dim_t k = 0; k < (dim_t)slice_mode; k++)
    below *= modes[k];
  for (dim_t k = slice_mode + 1; k < N; k++)
    above *= modes[k];
  std::vector<std::vector<double>> slab_store(W);
  double sumsq = 0.0;
  for (size_t r = 0; r < W; r++) {
    const dim_t ext = cuts[r + 1] - cuts[r];
    const double *src = X.get_data() + below * cuts[r];
    if (above > 1) {
      slab_store[r].resize(below * ext * above);
      for (dim_t u = 0; u < above; u++)
        std::copy(src + u * below * modes[slice_mode], src + u * below * modes[slice_mode] + below * ext,
                  slab_store[r].data() + u * below * ext);
      src = slab_store[r].data();
    }
    check(*eng[r], cals_b200_set_tensor_slab(eng[r]->ctx, (int)N, m64.data(), slice_mode, c64.data(), src),
          "cals_b200_set_tensor_slab");
  }
  for (size_t r = 0; r < W; r++) {
    double nrm = 0.0;
    check(*eng[r], cals_b200_tensor_norm(eng[r]->ctx, &nrm), "cals_b200_tensor_norm");
    sumsq += nrm * nrm;
  }
  const unsigned flags = (opt.force_max_iter ? CALS_B200_FORCE_MAX_ITER : 0u) |
                         (opt.always_evict_first ? CALS_B200_ALWAYS_EVICT_FIRST : 0u) |
                         (opt.nnls ? CALS_B200_NNLS : 0u);
  std::vector<const double *> in(N);
  for (size_t r = 0; r < W; r++) {
    check(*eng[r], cals_b200_set_tensor_norm(eng[r]->ctx, std::sqrt(sumsq)), "cals_b200_set_tensor_norm");
    check(*eng[r], cals_b200_configure(eng[r]->ctx, buffer, opt.max_iterations, opt.tol, flags), "cals_b200_configure");
    check(*eng[r], cals_b200_set_line_search(eng[r]->ctx, opt.line_search, opt.ls_method, opt.ls_interval, opt.ls_step),
          "cals_b200_set_line_search");
    check(*eng[r], cals_b200_set_timing(eng[r]->ctx, opt.timing), "cals_b200_set_timing");
    check(*eng[r], cals_b200_set_pair_node(eng[r]->ctx, opt.pair_node), "cals_b200_set_pair_node");
    check(*eng[r], cals_b200_clear_models(eng[r]->ctx), "cals_b200_clear_models");
    for (Ktensor *kt : models) {
      for (dim_t n = 0; n < N; n++)
        in[n] = kt->get_factor(n).get_data();
      check(*eng[r], cals_b200_enqueue_model(eng[r]->ctx, kt->get_components(), in.data(), -1, 0, nullptr),
            "cals_b200_enqueue_model");
    }
  }
  // the loops of all devices run side by side (they meet in every exchange)
  std::vector<cals_b200_report> reps(W);
  std::vector<std::string> errors(W);
  std::vector<std::thread> workers;
  for (size_t r = 0; r < W; r++)
    workers.emplace_back([&, r] {
      if (cals_b200_run(eng[r]->ctx, &reps[r]) != 0)
        errors[r] = cals_b200_last_error(eng[r]->ctx);
    });
  for (auto &w : workers)
    w.join();
  for (size_t r = 0; r < W; r++)
    if (!errors[r].empty())
      throw B200Error("cp_cals (sliced) on device " + std::to_string(devices[r]) + ": " + errors[r]);

  RunResult out;
  out.rep = reps[0];
  const size_t M = models.size();
  std::vector<double *> fptr(M * N), lptr(M);
  std::vector<cals_b200_model_stats> stats(M);
  for (size_t m = 0; m < M; m++) {
    for (dim_t n = 0; n < N; n++)
      fptr[m * N + n] = models[m]->get_factor(n).get_data();
    lptr[m] = models[m]->get_lambda().data();
  }
  check(*eng[0], cals_b200_fetch_all(eng[0]->ctx, fptr.data(), lptr.data(), stats.data()), "cals_b200_fetch_all");
  for (size_t m = 0; m < M; m++) {
    models[m]->set_iters(static_cast<dim_t>(stats[m].iters));
    models[m]->set_approximation_error(stats[m].error);
    models[m]->set_fit(stats[m].fit, stats[m].old_fit);
  }
  uint64_t n_it = 0;
  check(*eng[0], cals_b200_fetch_iteration_cols(eng[0]->ctx, nullptr, 0, &n_it), "cals_b200_fetch_iteration_cols");
  std::vector<uint32_t> c32(n_it);
  if (n_it)
    check(*eng[0], cals_b200_fetch_iteration_cols(eng[0]->ctx, c32.data(), n_it, &n_it), "fetch_iteration_cols");
  out.cols.assign(c32.begin(), c32.end());
  for (size_t r = 0; r < W; r++) // leave no peer mapping behind: the next call may use other devices
    check(*eng[r], cals_b200_comm_disconnect(eng[r]->ctx), "cals_b200_comm_disconnect");
  return out;
}

std::vector<std::vector<size_t>> shard_models(const std::vector<dim_t> &ranks, size_t n_parts) {
  // Largest rank first (ties: queue order), each model to the shard with the smallest sum of ranks so far (ties: lowest
  // shard index); inside a shard the queue order is kept.  Largest-first keeps the shards within one small rank of each
  // other -- the per-GPU column counts set the MTTKRP tile fill, and the slowest shard sets the time of the job.
  std::vector<std::vector<size_t>> parts(std::max<size_t>(n_parts, 1));
  std::vector<dim_t> load(parts.size(), 0);
  std::vector<size_t> order(ranks.size());
  std::iota(order.begin(), order.end(), size_t(0));
  std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return ranks[a] > ranks[b]; });
  for (size_t i : order) {
    size_t best = 0;
    for (size_t p = 1; p < parts.size(); p++)
      if (load[p] < load[best])
        best = p;
    parts[best].push_back(i);
    load[best] += ranks[i];
  }
  for (auto &p : parts)
    std::sort(p.begin(), p.end());
  return parts;
}

} // namespace detail

// ---------------------------------------------------------------------------------------------------------------------
static void reject_unsupported(update::UPDATE_METHOD um, bool line_search, ls::LS_METHOD lm, const char *who) {
  if (um != update::UNCONSTRAINED && um != update::NNLS)
    throw B200Error(std::string(who) + ": unknown update method");
  if (line_search && lm != ls::NO_ERROR_CHECKING && lm != ls::ERROR_CHECKING_SERIAL)
    throw B200Error(std::string(who) + ": line search method '" + ls::ls_method_names[lm] +
                    "' is not on the B200 path (the reference's own dispatcher ignores it too, "
                    "src/utils/line_search.cpp:228-259); there is no CPU fallback");
}

CalsReport cp_cals(const Tensor &X, KtensorQueue &kt_queue, CalsParams &cals_params) {
  reject_unsupported(cals_params.update_method, cals_params.line_search, cals_params.line_search_method, "cp_cals");
  if (X.get_n_modes() < 3)
    throw B200Error("cp_cals: tensors need at least 3 modes (the reference asserts the same, src/cals.cpp:52)");

  CalsReport rep;
  rep.tensor_rank = X.get_rank();
  rep.n_modes = X.get_n_modes();
  rep.modes = X.get_modes();
  rep.max_iter = cals_params.max_iterations;
  rep.n_threads = get_threads();
  rep.buffer_size = cals_params.buffer_size;
  rep.tol = cals_params.tol;
  rep.cuda = true;
  rep.update_method = cals_params.update_method;
  rep.line_search = cals_params.line_search;
  rep.line_search_interval = cals_params.line_search_interval;
  rep.line_search_step = cals_params.line_search_step;
  rep.line_search_method = cals_params.line_search_method;

  Timer total;
  total.start();

  // drain the queue (the reference pops every model it admits, src/cals.cpp:182-192)
  std::vector<Ktensor *> models;
  models.reserve(kt_queue.size());
  while (!kt_queue.empty()) {
    models.push_back(&kt_queue.front().get());
    kt_queue.pop();
  }

  detail::RunOptions opt;
  opt.buffer_size = cals_params.buffer_size;
  opt.max_iterations = cals_params.max_iterations;
  opt.tol = cals_params.tol;
  opt.force_max_iter = cals_params.force_max_iter;
  opt.always_evict_first = cals_params.always_evict_first;
  opt.nnls = cals_params.update_method == update::NNLS;
  opt.line_search = cals_params.line_search;
  opt.ls_method = static_cast<int>(cals_params.line_search_method);
  opt.ls_interval = cals_params.line_search_interval;
  opt.ls_step = cals_params.line_search_step;
  opt.timing = cals_params.timing;
  opt.pair_node = cals_params.mttkrp_method != mttkrp::MTTKRP_METHOD::MTTKRP;

  std::vector<int> devices = cals_params.devices.empty() ? std::vector<int>{0} : cals_params.devices;
  rep.n_devices = static_cast<int>(devices.size());

  std::vector<detail::RunResult> results(devices.size());
  if (cals_params.slice_mode >= 0 && devices.size() > 1) {
    results.resize(1);
    results[0] = detail::run_sliced(devices, cals_params.slice_mode, X, models, opt);
  } else if (devices.size() == 1) {
    results[0] = detail::run_on_device(devices[0], X, models, opt);
  } else {
    std::vector<dim_t> ranks(models.size());
    for (size_t i = 0; i < models.size(); i++)
      ranks[i] = models[i]->get_components();
    const auto parts = detail::shard_models(ranks, devices.size());
    std::vector<std::thread> workers;
    std::vector<std::string> errors(devices.size());
    for (size_t d = 0; d < devices.size(); d++)
      workers.emplace_back([&, d] {
        try {
          std::vector<Ktensor *> mine;
          for (size_t i : parts[d])
            mine.push_back(models[i]);
          results[d] = detail::run_on_device(devices[d], X, mine, opt);
        } catch (const std::exception &ex) {
          errors[d] = ex.what();
        }
      });
    for (auto &w : workers)
      w.join();
    for (size_t d = 0; d < devices.size(); d++)
      if (!errors[d].empty())
        throw B200Error("cp_cals on device " + std::to_string(devices[d]) + ": " + errors[d]);
  }
  total.stop();

  // merge the per-device reports: iteration i of the job = iteration i of every shard, side by side
  for (const auto &r : results) {
    rep.iter = std::max<dim_t>(rep.iter, r.rep.iter);
    rep.n_ktensors += static_cast<int>(r.rep.n_ktensors);
    rep.ktensor_comp_sum += static_cast<int>(r.rep.ktensor_comp_sum);
    if (r.rep.x_norm > 0)
      rep.X_norm = r.rep.x_norm;
    rep.device_ms = std::max(rep.device_ms, r.rep.device_ms);
    rep.mttkrp_ms = std::max(rep.mttkrp_ms, r.rep.mttkrp_ms);
    rep.update_ms = std::max(rep.update_ms, r.rep.update_ms);
    rep.kernel_launches += r.rep.kernel_launches;
    rep.mttkrp_flops += r.rep.mttkrp_flops;
    rep.ls_performed += r.ls_performed;
    rep.ls_failed += r.ls_failed;
  }
  if (models.empty())
    rep.X_norm = X.norm();
  rep.total_time = total.get_time();

  const dim_t its = rep.iter;
  rep.cols.assign(its, 0);
  for (const auto &r : results)
    for (dim_t i = 0; i < r.cols.size() && i < its; i++)
      rep.cols[i] += r.cols[i];
  rep.flops_per_iteration.assign(its, 0);
  for (dim_t i = 0; i < its; i++)
    rep.flops_per_iteration[i] = 2ull * rep.n_modes * X.get_n_elements() * rep.cols[i];

  rep.als_times = Matrix(AlsTimers::LENGTH, std::max<dim_t>(its, 1));
  rep.mode_times = Matrix(ModeTimers::LENGTH * rep.n_modes, std::max<dim_t>(its, 1));
  rep.mttkrp_times = Matrix(MttkrpTimers::LENGTH * rep.n_modes, std::max<dim_t>(its, 1));
  rep.als_times.zero();
  rep.mode_times.zero();
  rep.mttkrp_times.zero();
  for (dim_t i = 0; i < its; i++) {
    rep.als_times(AlsTimers::ITERATION, i) = rep.device_ms * 1e-3 / static_cast<double>(its);
    for (dim_t n = 0; n < rep.n_modes; n++) {
      rep.mode_times(n * ModeTimers::LENGTH + ModeTimers::MTTKRP, i) =
          rep.mttkrp_ms * 1e-3 / static_cast<double>(its * rep.n_modes);
      rep.mode_times(n * ModeTimers::LENGTH + ModeTimers::UPDATE, i) =
          rep.update_ms * 1e-3 / static_cast<double>(its * rep.n_modes);
    }
  }
  return rep;
}

// ---------------------------------------------------------------------------------------------------------------------
JKReport jk_cp_cals(const Tensor &X, vector<Ktensor> &kt_vector, CalsParams &cals_params) {
  vector<Ktensor> bases(kt_vector);
  for (Ktensor &b : bases)
    b.denormalize().normalize();

  Timer pre, run;
  pre.start();
  vector<vector<Ktensor>> jk_input(bases.size());
  for (size_t b = 0; b < bases.size(); b++)
    utils::generate_jk_ktensors(bases[b], jk_input[b]);
  KtensorQueue queue;
  for (auto &group : jk_input)
    for (Ktensor &m : group)
      queue.emplace(m);
  pre.stop();

  run.start();
  cp_cals(X, queue, cals_params);
  run.stop();

  // reference src/cals.cpp:431-437
  for (auto &group : jk_input)
    for (Ktensor &m : group) {
      m.set_jk_fiber(0.0);
      m.denormalize();
      m.normalize();
      m.set_jk_fiber(NAN);
    }
  for (size_t b = 0; b < bases.size(); b++)
    utils::jk_permutation_adjustment(bases[b], jk_input[b]);

  return JKReport{JKTime{pre.get_time(), run.get_time()}, std::move(jk_input)};
}

// ---------------------------------------------------------------------------------------------------------------------
std::vector<double> core_consistency(const Tensor &X, const std::vector<Ktensor> &models, int device) {
  detail::EngineHandle &e = detail::engine_for_device(device);
  std::lock_guard<std::mutex> lk(e.mu);
  const size_t M = models.size();
  std::vector<double> cc(M);
  if (M == 0)
    return cc;
  detail::upload_tensor(e, X, false);
  const dim_t N = X.get_n_modes();
  // lambda folded into mode 0 (the engine takes lambda = 1 for enqueued models)
  std::vector<std::vector<double>> first(M);
  std::vector<const double *> in(M * N);
  std::vector<uint64_t> ranks(M);
  std::vector<int> jk_modes(M);
  std::vector<int64_t> jk_fibers(M);
  for (size_t m = 0; m < M; m++) {
    const Ktensor &kt = models[m];
    if (kt.get_n_modes() != N)
      throw B200Error("core_consistency: a Ktensor has a different number of modes than the tensor");
    const dim_t R = kt.get_components();
    for (dim_t n = 0; n < N; n++) {
      if (kt.get_factor(n).get_rows() != X.get_modes()[n])
        throw B200Error("core_consistency: a Ktensor factor does not match the tensor extents");
      in[m * N + n] = kt.get_factor(n).get_data();
    }
    const Matrix &F0 = kt.get_factor(0);
    const dim_t rows = F0.get_rows();
    const std::vector<double> &lam = kt.get_lambda();
    first[m].assign(F0.get_data(), F0.get_data() + rows * R);
    for (dim_t j = 0; j < R && j < lam.size(); j++)
      for (dim_t i = 0; i < rows; i++)
        first[m][i + j * rows] *= lam[j];
    in[m * N] = first[m].data();
    ranks[m] = R;
    jk_modes[m] = kt.is_jk() ? (int)kt.get_jk_mode() : -1;
    jk_fibers[m] = kt.is_jk() ? (int64_t)kt.get_jk_fiber() : 0;
  }
  // the pooled context keeps the buffer size of its last run; batches of the default size (cp_cals configures again)
  const dim_t buffer = std::max<dim_t>(4200, *std::max_element(ranks.begin(), ranks.end()));
  detail::check(e, cals_b200_configure(e.ctx, buffer, 200, 1e-7, 0u), "cals_b200_configure");
  detail::check(e, cals_b200_clear_models(e.ctx), "cals_b200_clear_models");
  detail::check(e, cals_b200_enqueue_models(e.ctx, M, ranks.data(), in.data(), jk_modes.data(), jk_fibers.data()),
                "cals_b200_enqueue_models");
  detail::check(e, cals_b200_core_consistency(e.ctx, cc.data(), nullptr), "cals_b200_core_consistency");
  return cc;
}

// ---------------------------------------------------------------------------------------------------------------------
void CalsParams::print() const {
  using std::cout;
  using std::endl;
  const char *rule = "---------------------------------------";
  cout << rule << "\nCALS parameters\n" << rule << endl;
  cout << "Tol:             " << tol << endl;
  cout << "Max Iterations:  " << max_iterations << endl;
  cout << "Buffer Size:     " << buffer_size << endl;
  cout << "Mttkrp Method:   " << mttkrp::mttkrp_method_names[mttkrp_method] << " (MTTKRP: one contraction per mode; otherwise shared where possible)" << endl;
  cout << "Update Method:   " << update::update_method_names[update_method] << endl;
  cout << "Line Search:     " << (line_search ? "true" : "false") << endl;
  if (line_search) {
    cout << "-Line Search Interval: " << line_search_interval << " iterations" << endl;
    cout << "-Line Search Method:   " << ls::ls_method_names[line_search_method] << endl;
  }
  cout << "CUDA:            true (B200, devices:";
  if (devices.empty())
    cout << " 0";
  for (int d : devices)
    cout << " " << d;
  cout << ")" << endl << rule << endl;
}

// CSV layout of the reference (include/cals.h:70-132): one header line, then one line per CALS iteration.
void CalsReport::print_header(const std::string &file_name, const std::string &sep) const {
  std::ofstream file(file_name, std::ios::out);
  for (const char *name : {"TENSOR_RANK", "TENSOR_MODES", "BUFFER_SIZE", "N_KTENSORS", "KTENSOR_COMP_SUM",
                           "UPDATE_METHOD", "LINE_SEARCH", "MAX_ITERS", "ITER", "NUM_THREADS", "TOTAL", "FLOPS", "COLS"})
    file << name << sep;
  AlsTimers at;
  ModeTimers mt;
  for (const auto &name : at.names)
    file << name << sep;
  for (dim_t n = 0; n < modes.size(); n++)
    for (const auto &name : mt.names)
      file << "MODE_" << n << "_" << name << sep;
  file << std::endl;
}

void CalsReport::print_to_file(const std::string &file_name, const std::string &sep) const {
  std::ofstream file(file_name, std::ios::app);
  for (dim_t it = 0; it < iter; it++) {
    file << tensor_rank << sep << utils::mode_string(modes) << sep << buffer_size << sep << n_ktensors << sep
         << ktensor_comp_sum << sep << update::update_method_names[update_method] << sep << line_search << sep
         << max_iter << sep << it + 1 << sep << n_threads << sep << total_time << sep;
    file << flops_per_iteration[it] << sep << cols[it] << sep;
    file << std::scientific;
    for (dim_t i = 0; i < als_times.get_rows(); i++)
      file << als_times(i, it) << sep;
    for (dim_t i = 0; i < mode_times.get_rows(); i++)
      file << mode_times(i, it) << sep;
    file << std::defaultfloat << std::endl;
  }
}

} // namespace cals
