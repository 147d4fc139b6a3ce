// cals::cp_cals / cals::jk_cp_cals -- the drop-in C++ surface of the B200 path (reference include/cals.h:20-198).
//
//   CalsReport cp_cals(const Tensor &X, KtensorQueue &kt_queue, CalsParams &cals_params);     reference src/cals.cpp:19
//   JKReport jk_cp_cals(const Tensor &X, vector<Ktensor> &kt_vector, CalsParams &cals_params); reference src/cals.cpp:397
//
// Host code here is a thin layer: it hands X and the queued models to the C ABI (include/cals_b200.h), where the whole
// do/while loop of the reference runs on the device, and writes the fitted models back into the caller's Ktensors.
// There is no CPU implementation behind these functions: without a B200 they throw cals::B200Error.
#ifndef CALS_B200_CALS_H
#define CALS_B200_CALS_H

#include <cfloat>
#include <functional>
#include <queue>
#include <stdexcept>
#include <string>
#include <vector>

#include "als.h"
#include "ktensor.h"
#include "tensor.h"
#include "timer.h"
#include "utils/line_search.h"
#include "utils/mttkrp.h"
#include "utils/update.h"
#include "utils/utils.h"

namespace cals {

// Raised for everything the reference answers with `std::cerr << ...; exit(EXIT_FAILURE)` / abort(): unsupported
// options (the line-search method the reference never dispatches), a missing device, a failed CUDA call.  Uncaught,
// it terminates the process like the reference does; caught, it lets a host application recover.
struct B200Error : std::runtime_error {
  using std::runtime_error::runtime_error;
};

typedef std::queue<std::reference_wrapper<Ktensor>> KtensorQueue;

struct CalsReport {
  // target tensor
  int tensor_rank{0};
  dim_t n_modes{0};
  vector<dim_t> modes;
  double X_norm{0.0};

  // execution parameters
  dim_t iter{0};
  dim_t max_iter{0};
  int n_threads{0};
  dim_t buffer_size{0};
  int n_ktensors{0};
  int ktensor_comp_sum{0};
  double tol{0.0};
  bool cuda{true};
  update::UPDATE_METHOD update_method{update::UNCONSTRAINED};
  std::string output_file_name;

  bool line_search{false};
  int line_search_interval{0};
  double line_search_step{0.0};
  dim_t ls_performed{0};
  dim_t ls_failed{0};
  ls::LS_METHOD line_search_method{ls::NO_ERROR_CHECKING};

  double total_time{0.0};
  // Per-iteration tables with the reference's layout (rows = timers, columns = iterations).  The B200 loop runs
  // without host synchronisation, so per-iteration host timers do not exist: ITERATION holds the device time of the
  // whole loop divided by the iteration count, the others 0 (see the device_* fields for measured numbers).
  Matrix als_times{};
  Matrix mode_times{};
  Matrix mttkrp_times{};
  vector<uint64_t> flops_per_iteration; // 2 * N * nX * cols[it]
  vector<dim_t> cols;                   // active multi-factor columns in every iteration

  // extensions: what the engine measured (cals_b200_report)
  int n_devices{1};
  double device_ms{0.0};
  double mttkrp_ms{0.0};
  double update_ms{0.0};
  uint64_t kernel_launches{0};
  double mttkrp_flops{0.0};

  void print_header(const std::string &file_name, const std::string &sep = ";") const;
  void print_to_file(const std::string &file_name, const std::string &sep = ";") const;
};

struct CalsParams {
  update::UPDATE_METHOD update_method{update::UPDATE_METHOD::UNCONSTRAINED};
  mttkrp::MTTKRP_METHOD mttkrp_method{mttkrp::MTTKRP_METHOD::AUTO}; // MTTKRP: one contraction per mode; else shared (pair node)
  cals::mttkrp::MttkrpLut mttkrp_lut{};                             // accepted, ignored

  dim_t max_iterations{200};
  double tol{1e-7};
  bool cuda{false}; // accepted; this library always runs on the B200
  dim_t buffer_size{4200};

  bool line_search{false};
  int line_search_interval{5};
  double line_search_step{0};
  ls::LS_METHOD line_search_method{ls::NO_ERROR_CHECKING};

  bool force_max_iter{false};
  bool always_evict_first{false};

  // extensions
  std::vector<int> devices{}; // CUDA ordinals to shard the model set over (X replicated); empty = {0}
  // >= 0: instead of sharding the models, slice X along this mode over `devices` (a tensor too large for one GPU,
  // BASELINE config 5): every device holds a slab of X and all models; partial MTTKRPs are combined over NVLink peer
  // memory by the engine's exchange kernel.  -1 (default): replicate X, shard the models.
  int slice_mode{-1};
  int timing{0};              // 1: bracket MTTKRP / update kernels with CUDA events (fills mttkrp_ms / update_ms)

  void print() const;
};

CalsReport cp_cals(const Tensor &X, KtensorQueue &kt_queue, CalsParams &cals_params);

JKReport jk_cp_cals(const Tensor &X, vector<Ktensor> &kt_vector, CalsParams &cals_params);

// Extension (no reference counterpart): the core consistency diagnostic (CORCONDIA, Bro & Kiers, J. Chemometrics 17
// (2003) 274-286) of every model against X, computed on one device.  Lambda is folded into mode 0; a jackknife model
// leaves out its row of mode 0.  3- and 4-mode tensors; NaN for a model of rank above the limit (96 for 3 modes, 64 for
// 4) or with a rank-deficient factor.
std::vector<double> core_consistency(const Tensor &X, const std::vector<Ktensor> &models, int device = 0);

} // namespace cals
#endif
