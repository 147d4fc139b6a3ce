// Host-only checks of the cals:: containers (no device needed): Tensor / Matrix / Ktensor bookkeeping, normalisation
// identities, jackknife helpers, linear sum assignment, the model sharding plan.  Prints OK and exits 0 on success.
// Usage: host_containers_check [DIR]  -- DIR (default /tmp) holds the scratch files of the file-format checks.
#include <cmath>
#include <cstdio>
#include <fstream>
#include <sstream>
#include <numeric>
#include <random>

#include "cals.h"
#include "multi_ktensor.h"
#include "utils/error.h"

#define REQUIRE(c)                                                                                                     \
  do {                                                                                                                 \
    if (!(c)) {                                                                                                        \
      std::printf("FAILED %s:%d: %s\n", __FILE__, __LINE__, #c);                                                       \
      return 1;                                                                                                        \
    }                                                                                                                  \
  } while (0)

namespace cals::detail {
std::vector<std::vector<size_t>> shard_models(const std::vector<dim_t> &ranks, size_t n_parts);
}

int main(int argc, char **argv) {
  using namespace cals;
  const std::string scratch = argc > 1 ? argv[1] : "/tmp";
  std::mt19937 gen(0);
  std::uniform_real_distribution<double> dist(-1.0, 1.0);
  auto draw = [&] { return dist(gen); };

  // Tensor: layout, views, copies, unfolding geometry
  Tensor T(std::vector<dim_t>{4, 3, 2});
  T.fill(draw);
  REQUIRE(T.get_n_elements() == 24 && T.get_n_modes() == 3 && !T.is_view());
  Tensor V(std::vector<dim_t>{4, 3, 2}, T.get_data());
  REQUIRE(V.is_view() && V.get_data() == T.get_data());
  Tensor Tc(T);
  REQUIRE(Tc.get_data() != T.get_data() && Tc[5] == T[5]);
  double ss = 0;
  for (dim_t i = 0; i < 24; i++)
    ss += T[i] * T[i];
  REQUIRE(std::fabs(T.norm() - std::sqrt(ss)) < 1e-14);
  Unfolding u0 = T.implicit_unfold(0), u1 = T.implicit_unfold(1), u2 = T.implicit_unfold(2);
  REQUIRE(u0.n_blocks == 1 && u0.rows == 4 && u0.cols == 6);
  REQUIRE(u1.n_blocks == 2 && u1.rows == 3 && u1.cols == 4 && u1.block_offset == 12);
  REQUIRE(u2.n_blocks == 1 && u2.rows == 2 && u2.cols == 12);

  // Matrix
  Matrix M(3, 2);
  M.fill(draw);
  REQUIRE(M(2, 1) == M.get_data()[5] && M.get_col_stride() == 3);
  Matrix Mt(2, 3);
  Mt.transpose_copy(M); // Mt holds the row-major image of M
  REQUIRE(Mt.get_data()[1 + 2 * 2] == M(2, 1));

  // Ktensor: fill + normalise, reconstruction invariance under denormalize/normalize
  Ktensor K(3, {5, 4, 6});
  K.fill(draw);
  for (dim_t n = 0; n < 3; n++)
    for (dim_t c = 0; c < 3; c++) {
      double s = 0;
      for (dim_t r = 0; r < K.get_factor(n).get_rows(); r++)
        s += K.get_factor(n)(r, c) * K.get_factor(n)(r, c);
      REQUIRE(std::fabs(s - 1.0) < 1e-13);
    }
  Tensor R0 = K.to_tensor();
  K.denormalize().normalize();
  Tensor R1 = K.to_tensor();
  double gap = 0;
  for (dim_t i = 0; i < R0.get_n_elements(); i++)
    gap = std::max(gap, std::fabs(R0[i] - R1[i]));
  REQUIRE(gap < 1e-13);
  // signed max-abs normalisation of later iterations: lambda = entry of largest magnitude, first index on ties
  Ktensor S(1, {4, 3, 3});
  S.get_factor(0)(0, 0) = 0.5, S.get_factor(0)(1, 0) = -2.0, S.get_factor(0)(2, 0) = 2.0, S.get_factor(0)(3, 0) = 1.0;
  S.normalize(0, 2);
  REQUIRE(S.get_lambda()[0] == -2.0 && S.get_factor(0)(1, 0) == 1.0 && S.get_factor(0)(2, 0) == -1.0);
  // copies get new ids, copy() keeps the id
  Ktensor K2(K);
  REQUIRE(K2.get_id() != K.get_id() && K2.get_components() == 3);
  const int id2 = K2.get_id();
  K2.copy(K);
  REQUIRE(K2.get_id() == id2);

  // jackknife helpers
  std::vector<Ktensor> jk;
  utils::generate_jk_ktensors(K, jk);
  REQUIRE(jk.size() == 5 && jk[3].is_jk() && jk[3].get_jk_fiber() == 3 && jk[3].get_jk_mode() == 0);
  jk[3].set_jk_fiber(0.0);
  REQUIRE(jk[3].get_factor(0)(3, 1) == 0.0);
  Ktensor reg = jk[3].to_regular();
  REQUIRE(reg.get_factor(0).get_rows() == 4 && reg.get_factor(0)(3, 2) == jk[3].get_factor(0)(4, 2));
  jk[3].set_jk_fiber(NAN);
  REQUIRE(std::isnan(jk[3].get_factor(0)(3, 0)));
  // permutation adjustment: a leave-one-out model whose components are a permutation of the base model's.  The
  // reference applies new[:, c] = old[:, p[c]] with p[c] = base component matched to component c (src/utils/utils.cpp:
  // 88-99), which undoes the permutation when it is its own inverse -- a swap here.
  std::vector<Ktensor> shuffled;
  shuffled.emplace_back(K);
  const dim_t perm[3] = {2, 1, 0};
  for (dim_t n = 0; n < 3; n++)
    for (dim_t c = 0; c < 3; c++)
      for (dim_t r = 0; r < K.get_factor(n).get_rows(); r++)
        shuffled[0].get_factor(n)(r, c) = K.get_factor(n)(r, perm[c]);
  utils::jk_permutation_adjustment(K, shuffled);
  for (dim_t n = 0; n < 3; n++)
    for (dim_t e = 0; e < K.get_factor(n).get_n_elements(); e++)
      REQUIRE(shuffled[0].get_factor(n)[e] == K.get_factor(n)[e]);

  // linear sum assignment against brute force
  for (int trial = 0; trial < 20; trial++) {
    const dim_t n = 5;
    std::vector<double> cost(n * n);
    for (double &c : cost)
      c = draw();
    std::vector<int64_t> assign;
    utils::linear_sum_assignment(n, cost.data(), true, assign);
    double got = 0;
    for (dim_t i = 0; i < n; i++)
      got += cost[i * n + assign[i]];
    std::vector<int> p(n);
    std::iota(p.begin(), p.end(), 0);
    double best = -1e300;
    do {
      double s = 0;
      for (dim_t i = 0; i < n; i++)
        s += cost[i * n + p[i]];
      best = std::max(best, s);
    } while (std::next_permutation(p.begin(), p.end()));
    REQUIRE(std::fabs(got - best) < 1e-12);
  }

  // fast error == explicit error on the host helpers
  {
    Ktensor A(2, {4, 3, 5});
    A.fill(draw);
    Tensor X = A.to_tensor();
    std::vector<Matrix> grams;
    for (dim_t n = 0; n < 3; n++)
      grams.emplace_back(2, 2);
    ops::update_gramians(A, grams);
    ops::hadamard_all(grams);
    // G_last = X_(2) * KRP(A1, A0) = A2 * diag(lambda) * hadamard(gram0, gram1) for an exact model
    Matrix G(5, 2);
    std::vector<Matrix> g01;
    g01.emplace_back(2, 2);
    g01.emplace_back(2, 2);
    ops::update_gramian(A.get_factor(0), g01[0]);
    ops::update_gramian(A.get_factor(1), g01[1]);
    g01[0].hadamard(g01[1]);
    for (dim_t i = 0; i < 5; i++)
      for (dim_t c = 0; c < 2; c++) {
        double s = 0;
        for (dim_t r = 0; r < 2; r++)
          s += A.get_factor(2)(i, r) * A.get_lambda()[r] * g01[0](r, c);
        G(i, c) = s;
      }
    const double e = error::compute_fast_error(X.norm(), A.get_lambda(), A.get_factor(2), G, grams[0]);
    REQUIRE(e < 1e-6 * X.norm()); // the formula is a cancellation: ~sqrt(eps) * ||X||
    Matrix w1, w2;
    REQUIRE(error::compute_error(X, A, w1, w2) < 1e-13 * X.norm());
  }

  // sharding plan: every model exactly once, queue order kept inside a shard, loads balanced
  {
    std::vector<dim_t> ranks;
    for (dim_t r = 1; r <= 20; r++)
      ranks.insert(ranks.end(), 10, r);
    auto parts = detail::shard_models(ranks, 8);
    std::vector<int> seen(ranks.size(), 0);
    dim_t lo = ~dim_t(0), hi = 0;
    for (auto &p : parts) {
      dim_t load = 0;
      for (size_t k = 0; k < p.size(); k++) {
        seen[p[k]]++;
        load += ranks[p[k]];
        REQUIRE(k == 0 || p[k] > p[k - 1]);
      }
      lo = std::min(lo, load), hi = std::max(hi, load);
    }
    for (int s : seen)
      REQUIRE(s == 1);
    REQUIRE(hi - lo <= 2); // largest rank first
  }

  // MultiKtensor: first-fit placement, BufferFull, detach on removal, stable compaction (reference
  // src/multi_ktensor.cpp:14-39,41-130,132-163,188-264)
  {
    std::vector<dim_t> modes{4, 3, 5};
    MultiKtensor mk(modes, 10);
    REQUIRE(mk.get_factor(0).get_cols() == 0 && mk.get_leftmost_id() == 0);
    std::vector<Ktensor> ms;
    for (dim_t r : {3, 2, 4})
      ms.emplace_back(r, modes);
    for (Ktensor &m : ms)
      m.fill(draw);
    std::vector<Ktensor> orig(ms);
    for (Ktensor &m : ms)
      mk.add(m);
    REQUIRE(mk.get_factor(1).get_cols() == 9 && mk.get_registry().size() == 3 && mk.get_leftmost_id() == 1);
    REQUIRE(mk.get_registry().at(2).col == 3 && ms[1].get_iters() == 1);
    // the models now live in the buffer: same values, storage inside the multi-factor
    REQUIRE(ms[1].get_factor(2).get_data() == mk.get_factor(2).get_data() + 3 * 5);
    REQUIRE(mk.get_factor(2)(4, 4) == orig[1].get_factor(2)(4, 1));
    // Gramians of the incoming factors
    REQUIRE(std::fabs(mk.get_registry().at(3).gramians[0](2, 2) - 1.0) < 1e-13);
    Ktensor big(2, modes);
    big.fill(draw);
    bool full = false;
    try {
      mk.add(big); // only one free column
    } catch (BufferFull &) {
      full = true;
    }
    REQUIRE(full);
    // write through the buffer, remove the middle model: it takes the value home, its columns are zeroed
    mk.get_factor(0)(1, 3) = 42.0;
    mk.remove(2);
    REQUIRE(ms[1].get_factor(0)(1, 0) == 42.0 && ms[1].get_factor(0).get_data() != mk.get_factor(0).get_data() + 12);
    REQUIRE(mk.get_factor(0)(1, 3) == 0.0 && mk.get_registry().count(2) == 0);
    mk.add(big); // first fit: the hole left by the rank-2 model
    REQUIRE(mk.get_registry().at(4).col == 3);
    mk.remove(1);
    REQUIRE(mk.get_leftmost_id() == 0 && mk.get_factor(0).get_cols() == 9);
    mk.compress(); // [., ., ., big, big, m3 x4] -> [big, big, m3 x4]
    REQUIRE(mk.get_factor(0).get_cols() == 6 && mk.get_registry().at(4).col == 0 && mk.get_registry().at(3).col == 2);
    REQUIRE(mk.get_leftmost_id() == 4);
    for (dim_t e = 0; e < ms[2].get_factor(1).get_n_elements(); e++)
      REQUIRE(ms[2].get_factor(1)[e] == orig[2].get_factor(1)[e]);
    REQUIRE(ms[2].get_factor(1).get_data() == mk.get_factor(1).get_data() + 2 * 3);
    REQUIRE(mk.get_factor(1).get_data()[6 * 3] == 0.0); // vacated columns are clean
    mk.remove(3);
    mk.remove(4);
    REQUIRE(mk.get_factor(0).get_cols() == 0 && mk.get_registry().empty());
  }

  // text tensor files (reference src/tensor.cpp:35-65: extents on the first line, values in column-major order)
  {
    const std::string path = scratch + "/cals_b200_tensor_check.txt";
    {
      std::ofstream f(path);
      f << "3 2 2\n";
      for (int i = 0; i < 12; i++)
        f << (i * 0.5 - 1.25) << (i % 4 == 3 ? "\n" : " ");
    }
    Tensor F{path};
    REQUIRE(F.get_n_modes() == 3 && F.get_modes()[0] == 3 && F.get_modes()[2] == 2 && F.get_n_elements() == 12);
    REQUIRE(F[0] == -1.25 && F[7] == 2.25 && F[11] == 4.25);
    bool threw = false;
    try {
      Tensor missing{scratch + "/cals_b200_no_such_file.txt"};
    } catch (const std::exception &) {
      threw = true;
    }
    REQUIRE(threw);
    std::remove(path.c_str());
  }

  // report CSV writers keep the reference's column set (include/cals.h:70-132, include/als.h:70-135)
  {
    CalsReport rep;
    rep.modes = {4, 3, 5};
    rep.n_modes = 3;
    rep.iter = 2;
    rep.max_iter = 7;
    rep.buffer_size = 9;
    rep.n_ktensors = 3;
    rep.ktensor_comp_sum = 6;
    rep.n_threads = 4;
    rep.total_time = 0.5;
    rep.flops_per_iteration = {10, 20};
    rep.cols = {6, 4};
    rep.als_times = Matrix(AlsTimers::LENGTH, 2);
    rep.mode_times = Matrix(ModeTimers::LENGTH * 3, 2);
    rep.als_times.zero();
    rep.mode_times.zero();
    const std::string path = scratch + "/cals_b200_report_check.csv";
    rep.print_header(path);
    rep.print_to_file(path);
    std::ifstream f(path);
    std::string header, l1, l2, extra;
    std::getline(f, header);
    std::getline(f, l1);
    std::getline(f, l2);
    REQUIRE(header.rfind("TENSOR_RANK;TENSOR_MODES;BUFFER_SIZE;N_KTENSORS;KTENSOR_COMP_SUM;UPDATE_METHOD;LINE_SEARCH;"
                         "MAX_ITERS;ITER;NUM_THREADS;TOTAL;FLOPS;COLS;ITERATION;DEFRAGMENTATION;ERROR;LINESEARCH;G_COPY;"
                         "MODE_0_TOTAL_MTTKRP;MODE_0_UPDATE;", 0) == 0);
    REQUIRE(l1.rfind("0;4-3-5;9;3;6;unconstrained;0;7;1;4;0.5;10;6;", 0) == 0);
    REQUIRE(l2.rfind("0;4-3-5;9;3;6;unconstrained;0;7;2;4;0.5;20;4;", 0) == 0);
    REQUIRE(!std::getline(f, extra));
    auto fields = [](const std::string &line) { return std::count(line.begin(), line.end(), ';'); };
    REQUIRE(fields(header) == fields(l1) && fields(header) == 13 + 5 + 6);
    std::remove(path.c_str());

    AlsReport ar;
    ar.modes = {4, 3, 5};
    ar.n_modes = 3;
    ar.iter = 3;
    ar.max_iter = 5;
    ar.ktensor_id = 17;
    ar.ktensor_components = 2;
    ar.als_times = Matrix(AlsTimers::LENGTH, 5);
    ar.mode_times = Matrix(ModeTimers::LENGTH * 3, 5);
    ar.als_times.zero();
    ar.mode_times.zero();
    ar.print_header(path);
    ar.print_to_file(path);
    std::ifstream g(path);
    std::getline(g, header);
    std::getline(g, l1);
    REQUIRE(header.rfind("TENSOR_RANK;TENSOR_MODES;KTENSOR_ID;KTENSOR_COMP;UPDATE_METHOD;LINE_SEARCH;MAX_ITERS;ITER;"
                         "NUM_THREADS;TOTAL;FLOPS;ITERATION;", 0) == 0);
    REQUIRE(l1.rfind("0;4-3-5;17;2;unconstrained;0;5;3;", 0) == 0 && fields(header) == fields(l1));
    std::remove(path.c_str());
  }

  set_threads(6);
  REQUIRE(get_threads() == 6);
  std::printf("OK\n");
  return 0;
}
