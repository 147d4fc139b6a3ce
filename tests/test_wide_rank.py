"""Models above the shared-memory update kernel's rank bound (96 unconstrained): the multi-CTA update path of
cp-cals_b200/csrc/wide.cuh, against the oracle and against the rest of the engine (-m gpu)."""
import os
import subprocess

import numpy as np
import pytest

import caseio
import oracle
from helpers import assert_models_close, to_ktensors

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _tensor(rng, modes, true_rank=8, noise=0.1):
    gen = [rng.uniform(-1, 1, size=(i, true_rank)) for i in modes]
    return caseio.ktensor_to_tensor(gen, np.ones(true_rank)) + noise * rng.standard_normal(modes)


def _assert_moderate_conditioning(models, limit=1e10):
    """cond(H) of every mode from the oracle's fitted factors: a failure then points at the code, not at H."""
    for m in models:
        grams = [F.T @ F for F in m.factors]
        for n in range(len(grams)):
            H = np.ones_like(grams[0])
            for k, g in enumerate(grams):
                if k != n:
                    H = H * g
            c = np.linalg.cond(H)
            assert c < limit, "cond(H) = %.3e for rank %d, mode %d" % (c, m.factors[0].shape[1], n)


def _run_both(pkg, X, ranks, seed, K=3, buffer_size=None, rtol=1e-8, **kw):
    rng = np.random.default_rng(seed)
    ms = caseio.random_models(rng, X.shape, ranks)
    want = oracle.cp_cals(X, ms, max_iter=K, buffer_size=buffer_size, **kw)
    kts = to_ktensors(pkg, ms)
    p = pkg.CalsParams(max_iterations=K, buffer_size=buffer_size or sum(ranks),
                       force_max_iter=kw.get("force_max_iter", False),
                       always_evict_first=kw.get("always_evict_first", False), tol=kw.get("tol", 1e-7))
    rep = pkg.cp_cals(X, kts, p)
    assert rep.iter == want.iters
    _assert_moderate_conditioning(want.models)
    assert all(k.chol_info == 0 for k in kts)
    assert_models_close(kts, want.models, want.x_norm, rtol=rtol, what="ranks %s" % (ranks,))
    return kts, rep


@pytest.mark.parametrize("ranks", [[96, 97], [95, 97, 104, 3, 1]])
@pytest.mark.parametrize("K", [1, 2, 3, 4])
def test_ranks_straddling_the_bound(pkg, ranks, K):
    rng = np.random.default_rng(100 + K)
    X = _tensor(rng, (60, 55, 50))
    _run_both(pkg, X, ranks, seed=K, K=K, force_max_iter=True)


@pytest.mark.parametrize("rank", [128, 256, 512, 1024])
def test_large_ranks_vs_oracle(pkg, rank):
    rng = np.random.default_rng(rank)
    X = _tensor(rng, (60, 55, 50))
    _run_both(pkg, X, [rank], seed=rank, K=2, force_max_iter=True)


def test_four_mode_rank_160(pkg):
    rng = np.random.default_rng(160)
    X = _tensor(rng, (16, 14, 12, 10), true_rank=5)
    _run_both(pkg, X, [160, 7], seed=160, K=3, force_max_iter=True)


def test_queue_dynamics_across_wide_and_narrow(pkg):
    """A buffer narrower than the queue: admission, eviction and compaction move wide and narrow models alike."""
    rng = np.random.default_rng(7)
    X = _tensor(rng, (40, 36, 30))
    _run_both(pkg, X, [120, 5, 100, 30, 130, 2, 98], seed=7, K=3, buffer_size=260, force_max_iter=True)


def test_always_evict_first_with_wide_models(pkg):
    rng = np.random.default_rng(8)
    X = _tensor(rng, (40, 36, 30))
    _run_both(pkg, X, [110, 4, 100, 12], seed=8, K=4, buffer_size=230, force_max_iter=True, always_evict_first=True)


def test_tol_stopping_with_wide_models(pkg):
    """Unforced iterations: every model stops at the iteration the oracle stops at."""
    rng = np.random.default_rng(9)
    X = _tensor(rng, (40, 36, 30), true_rank=3, noise=0.01)
    _run_both(pkg, X, [100, 3, 120, 6], seed=9, K=12, buffer_size=230, tol=1e-4, rtol=1e-7)


def test_mttkrp_methods_agree(pkg):
    """Per-mode MTTKRP, the pair node and the multi-sweep schedule give the same wide-model results."""
    rng = np.random.default_rng(10)
    X = _tensor(rng, (72, 70, 66))
    ms = caseio.random_models(rng, X.shape, [130, 20, 97])
    out = {}
    for name, method, msdt in [("mttkrp", "mttkrp", "0"), ("pair", "auto", "0"), ("msdt", "auto", "1")]:
        os.environ["CALS_B200_MSDT"] = msdt
        try:
            with pkg.Engine(0) as eng:
                kts = to_ktensors(pkg, ms)
                pkg.cp_cals(X, kts, pkg.CalsParams(max_iterations=4, buffer_size=247, force_max_iter=True,
                                                   mttkrp_method=method), engine=eng)
        finally:
            del os.environ["CALS_B200_MSDT"]
        out[name] = kts
    for name in ("pair", "msdt"):
        for a, b in zip(out["mttkrp"], out[name]):
            for Fa, Fb in zip(a.factors, b.factors):
                assert np.linalg.norm(Fa - Fb) <= 1e-11 * np.linalg.norm(Fa), name


def test_jackknife_with_a_wide_base_model(pkg):
    """jk_cp_cals with a rank-110 base model: the leave-one-out models against the oracle."""
    rng = np.random.default_rng(11)
    modes = (12, 40, 36)
    X = _tensor(rng, modes)
    base = caseio.random_models(rng, modes, [110])[0]
    p = pkg.CalsParams(max_iterations=3, buffer_size=330, force_max_iter=True)
    rep, results = pkg.jk_cp_cals(X, [pkg.Ktensor(base.factors, base.lam)], p)
    bb = pkg.Ktensor(base.factors, base.lam).copy().denormalize().normalize()
    flat_in = [caseio.Model(factors=[F.copy() for F in bb.factors], lam=bb.lam.copy(), jk_mode=0, jk_fiber=i)
               for i in range(modes[0])]
    want = oracle.cp_cals(X, flat_in, max_iter=3, force_max_iter=True, buffer_size=330)
    assert rep.iter == want.iters
    for got, w in zip(results[0], want.models):
        wk = pkg.Ktensor([F.copy() for F in w.factors], w.lam.copy(), 0, w.jk_fiber)
        wk.set_jk_fiber(0.0)
        wk.denormalize().normalize()
        for n in range(1, 3):
            e = np.linalg.norm(got.factors[n] - wk.factors[n]) / np.linalg.norm(wk.factors[n])
            assert e <= 1e-8, (w.jk_fiber, n, e)


@pytest.mark.parametrize("method", ["no-error-checking", "error-checking-serial"])
def test_line_search_with_rank_300(pkg, method):
    rng = np.random.default_rng(12)
    X = _tensor(rng, (40, 38, 36))
    ms = caseio.random_models(rng, X.shape, [300, 5])
    K = 7
    want = oracle.cp_cals(X, ms, max_iter=K, force_max_iter=True, line_search=True,
                          ls_method=0 if method == "no-error-checking" else 1, ls_interval=3, ls_step=0.0)
    kts = to_ktensors(pkg, ms)
    rep = pkg.cp_cals(X, kts, pkg.CalsParams(max_iterations=K, buffer_size=305, force_max_iter=True,
                                             line_search=True, line_search_method=method, line_search_interval=3))
    assert rep.iter == want.iters
    assert_models_close(kts, want.models, want.x_norm, rtol=1e-8, what="line search " + method)


def test_singular_start_counts_chol_info(pkg):
    """A zero starting column gives H a zero pivot: chol_info counts it and the run completes, for the wide model as
    for a narrow one."""
    rng = np.random.default_rng(13)
    X = _tensor(rng, (40, 36, 30))
    ms = caseio.random_models(rng, X.shape, [120, 4])
    for m in ms:
        for F in m.factors:
            F[:, 1] = 0.0
    kts = to_ktensors(pkg, ms)
    rep = pkg.cp_cals(X, kts, pkg.CalsParams(max_iterations=2, buffer_size=124, force_max_iter=True))
    assert rep.iter == 2
    assert kts[0].chol_info > 0 and kts[1].chol_info > 0


def test_nnls_keeps_its_rank_bound(pkg):
    rng = np.random.default_rng(14)
    X = np.abs(_tensor(rng, (30, 28, 26)))
    ms = caseio.random_models(rng, X.shape, [81, 3])
    p = pkg.CalsParams(max_iterations=2, buffer_size=84, force_max_iter=True, update_method="nnls")
    with pytest.raises(pkg.CalsB200Error, match=r"model 0 has rank 81, above 80"):
        pkg.cp_cals(X, to_ktensors(pkg, ms), p)
    ms = caseio.random_models(rng, X.shape, [80, 3])
    want = oracle.cp_cals(X, ms, max_iter=2, force_max_iter=True, nnls=True)
    kts = to_ktensors(pkg, ms)
    pkg.cp_cals(X, kts, pkg.CalsParams(max_iterations=2, buffer_size=83, force_max_iter=True, update_method="nnls"))
    assert_models_close(kts, want.models, want.x_norm, rtol=1e-8, what="nnls rank 80")


def test_rerun_of_mixed_queue_is_bit_identical(pkg):
    rng = np.random.default_rng(15)
    X = _tensor(rng, (50, 40, 30))
    ms = caseio.random_models(rng, X.shape, [3, 200, 9, 97])
    with pkg.Engine(0) as eng:
        eng.set_tensor(X)
        eng.configure(309, 4, 1e-7, force_max_iter=True)
        eng.clear_models()
        eng.enqueue_many([m.factors for m in ms])
        eng.run()
        first = eng.fetch_all()
        eng.rerun()
        second = eng.fetch_all()
    for (fa, la, sa), (fb, lb, sb) in zip(first, second):
        for a, b in zip(fa, fb):
            assert np.array_equal(a, b)
        assert np.array_equal(la, lb)
        assert sa.error == sb.error


def test_driver_with_wide_models():
    exe = os.path.join(ROOT, "cp-cals_b200", "bin", "driver")
    out = subprocess.run([exe, "-t", "100-100-100", "-c", "97:100:2", "-i", "5"], capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0, out.stdout + out.stderr


CPP_PROGRAM = r"""
#include <cmath>
#include <cstdio>
#include <random>
#include "als.h"
#include "cals.h"
int main() {
  std::mt19937 gen(3);
  std::uniform_real_distribution<double> dist(-1.0, 1.0);
  auto src = [&] { return dist(gen); };
  cals::Ktensor P(6, {50, 45, 40});
  P.fill(src);
  cals::Tensor X = P.to_tensor();
  for (dim_t e = 0; e < X.get_n_elements(); e++)
    X[e] += 0.1 * src();
  cals::Ktensor start(128, {50, 45, 40});
  start.fill(src);
  cals::Ktensor a(start), b(start);
  cals::CalsParams cp;
  cp.max_iterations = 5;
  cp.force_max_iter = true;
  cp.buffer_size = 128;
  cals::KtensorQueue q;
  q.emplace(a);
  cals::cp_cals(X, q, cp);
  cals::AlsParams ap;
  ap.max_iterations = 5;
  ap.force_max_iter = true;
  ap.suppress_lut_warning = true;
  cals::cp_als(X, b, ap);
  cals::Tensor ta = a.to_tensor(), tb = b.to_tensor();
  const double na = ta.norm();
  for (dim_t e = 0; e < ta.get_n_elements(); e++)
    ta[e] -= tb[e];
  const double gap = ta.norm() / na;
  std::printf("rank 128: cp_cals vs cp_als relative gap %.3e, iterations %d %d\n", gap, (int)a.get_iters(),
              (int)b.get_iters());
  return (gap <= 1e-9 && a.get_iters() == b.get_iters()) ? 0 : 1;
}
"""


def test_cpp_cp_cals_and_cp_als_agree_at_rank_128(tmp_path):
    src = tmp_path / "wide_cpp.cpp"
    src.write_text(CPP_PROGRAM)
    exe = tmp_path / "wide_cpp"
    lib = os.path.join(ROOT, "cp-cals_b200")
    subprocess.run(["/usr/bin/g++", "-O1", "-std=c++17", "-I" + os.path.join(ROOT, "include"),
                    "-I" + os.path.join(ROOT, "include", "utils"), "-o", str(exe), str(src), "-L" + lib, "-lcals",
                    "-lcals_b200", "-pthread", "-Wl,-rpath," + lib], check=True, capture_output=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
