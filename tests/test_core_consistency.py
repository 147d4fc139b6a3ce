"""Core consistency (CORCONDIA, Bro & Kiers 2003) of every queued model: Engine.core_consistency / core_consistency /
cals::core_consistency (cp-cals_b200/csrc/corcon.cuh).

CPU part: the NumPy reference itself -- exact-Tucker data, invariance under column permutation and under scaling moved
between lambda and mode 0, and the planted rank-3 claim with the oracle's fitted models.
GPU part (-m gpu): the engine against that reference after runs, before runs, with jackknife sub-models, in several
batches, with per-model statuses, repeated calls, the absence of side effects and the C++ entry point.
"""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import caseio
import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------------------------------------------------
def corcondia_ref(X, factors, lam=None, jk_row=-1):
    """100 (1 - sum (G - I)^2 / R), G = X x_0 P_0^T .. x_{N-1} P_{N-1}^T, P_n = A_n (A_n^T A_n)^-1, A_0 = F_0 diag(lam)."""
    A = [np.array(F, dtype=np.float64) for F in factors]
    if lam is not None:
        A[0] = A[0] * np.asarray(lam)[None, :]
    if jk_row >= 0:
        A[0][jk_row, :] = 0.0
    P = [np.linalg.solve(a.T @ a, a.T).T for a in A]
    G = np.asarray(X, dtype=np.float64)
    for Pn in P:  # the leading axis is always the next mode; the r axes pile up at the end
        G = np.tensordot(G, Pn, axes=([0], [0]))
    R = A[0].shape[1]
    E = G.copy()
    idx = np.arange(R)
    E[(idx,) * len(A)] -= 1.0
    return 100.0 * (1.0 - float(np.sum(E * E)) / R)


def gram_conditions(factors, lam=None):
    A = [np.array(F, dtype=np.float64) for F in factors]
    if lam is not None:
        A[0] = A[0] * np.asarray(lam)[None, :]
    return [np.linalg.cond(a.T @ a) for a in A]


def tucker(core, A):
    X = core
    for a in A:  # contract the leading core axis with A_n; the new axis goes to the end
        X = np.tensordot(X, a, axes=([0], [1]))
    return X


def exact_tucker_case(rng, modes, R, eps):
    A = [rng.standard_normal((I, R)) for I in modes]
    E = eps * rng.standard_normal((R,) * len(modes))
    core = E.copy()
    idx = np.arange(R)
    core[(idx,) * len(modes)] += 1.0
    return tucker(core, A), A, 100.0 * (1.0 - float(np.sum(E * E)) / R)


def planted(rng, modes, R=3, noise=0.01):
    A = [rng.standard_normal((I, R)) for I in modes]
    X0 = caseio.ktensor_to_tensor(A, np.ones(R))
    N = rng.standard_normal(modes)
    return X0 + noise * np.linalg.norm(X0) / np.linalg.norm(N) * N


def close(got, want):
    return abs(got - want) <= 1e-8 * max(1.0, abs(want))


# ---- CPU: the reference ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("modes,R", [((9, 8, 7), 3), ((7, 6, 5, 4), 3), ((12, 10, 9), 5)])
def test_reference_exact_tucker(modes, R):
    rng = np.random.default_rng(R + len(modes))
    X, A, want = exact_tucker_case(rng, modes, R, 0.05)
    assert abs(corcondia_ref(X, A) - want) <= 1e-10


def test_reference_invariances():
    rng = np.random.default_rng(3)
    X = rng.standard_normal((10, 9, 8))
    F = [rng.standard_normal((I, 4)) for I in X.shape]
    lam = rng.uniform(0.5, 2.0, 4)
    base = corcondia_ref(X, F, lam)
    perm = np.array([2, 0, 3, 1])
    assert abs(corcondia_ref(X, [f[:, perm] for f in F], lam[perm]) - base) <= 1e-10 * max(1, abs(base))
    d = rng.uniform(0.5, 2.0, 4)  # scaling moved between lambda and mode 0
    assert abs(corcondia_ref(X, [F[0] * d, F[1], F[2]], lam / d) - base) <= 1e-10 * max(1, abs(base))
    assert abs(corcondia_ref(X, [F[0] * lam, F[1], F[2]]) - base) <= 1e-10 * max(1, abs(base))


def _planted_models(rng, X, ranks):
    ms = caseio.random_models(rng, X.shape, ranks)
    return ms, oracle.cp_cals(X, ms, max_iter=500, tol=1e-12)


def test_reference_planted_rank3_with_oracle():
    rng = np.random.default_rng(7)
    X = planted(rng, (30, 28, 26))
    ranks = [1, 2, 3, 3, 3, 5, 5, 5]
    _, res = _planted_models(rng, X, ranks)
    cc = [corcondia_ref(X, m.factors, m.lam) for m in res.models]
    assert all(c > 95 for c, r in zip(cc, ranks) if r <= 3), cc
    assert max(c for c, r in zip(cc, ranks) if r == 5) < min(c for c, r in zip(cc, ranks) if r == 3), cc


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _fit(pkg, X, ranks, seed, K, buffer_cols=None, jk=None, force=True):
    rng = np.random.default_rng(seed)
    ms = caseio.random_models(rng, X.shape, ranks)
    eng = pkg.Engine(0)
    eng.set_tensor(X)
    eng.configure(buffer_cols or sum(ranks), K, 1e-7, force_max_iter=force)
    eng.clear_models()
    eng.enqueue_many([m.factors for m in ms], jk)
    eng.run()
    return eng


def _check_against_reference(X, fitted, cc, status, jk=None):
    for i, (fs, lam, _) in enumerate(fitted):
        assert status[i] == 0, (i, status[i])
        assert max(gram_conditions(fs, lam)) < 1e6
        row = jk[i][1] if jk is not None and jk[i][0] == 0 else -1
        want = corcondia_ref(X, fs, lam, row)
        assert close(cc[i], want), (i, fs[0].shape[1], cc[i], want)


@pytest.mark.gpu
@pytest.mark.parametrize("modes,ranks", [
    ((37, 30, 26), list(range(1, 21))),           # odd fastest extent: the tensor goes through the staging block
    ((40, 33, 29), list(range(1, 21))),
    ((14, 12, 11, 10), list(range(1, 9))),
    ((160, 150, 140), [96, 20, 1]),
])
def test_after_run_against_numpy(pkg, modes, ranks):
    rng = np.random.default_rng(len(ranks) + modes[0])
    X = planted(rng, modes, R=5, noise=0.5)
    eng = _fit(pkg, X, ranks, seed=modes[1], K=4)
    cc, status = eng.core_consistency()
    _check_against_reference(X, eng.fetch_all(), cc, status)
    cc2, status2 = eng.core_consistency()
    assert np.array_equal(cc.view(np.int64), cc2.view(np.int64)) and np.array_equal(status, status2)
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("modes,R", [((21, 19, 17), 4), ((33, 30, 28), 12), ((9, 8, 7, 6), 3)])
def test_exact_tucker_without_run(pkg, modes, R):
    rng = np.random.default_rng(R)
    X, A, want = exact_tucker_case(rng, modes, R, 0.05)
    with pkg.Engine(0) as eng:
        eng.set_tensor(X)
        eng.clear_models()
        eng.enqueue_many([A, [a[:, ::-1] for a in A]])
        cc, status = eng.core_consistency()
    assert list(status) == [0, 0]
    assert close(cc[0], want) and close(cc[1], want), (cc, want)
    # the module-level entry point: lambda folded into mode 0
    kt = pkg.Ktensor([A[0] / 2.0] + A[1:], np.full(R, 2.0))
    got = pkg.core_consistency(X, [kt])
    assert close(got[0], want), (got, want)


@pytest.mark.gpu
def test_planted_rank3(pkg):
    rng = np.random.default_rng(7)
    X = planted(rng, (30, 28, 26))
    ranks = [1, 2, 3, 3, 3, 5, 5, 5]
    ms = caseio.random_models(rng, X.shape, ranks)
    kts = [pkg.Ktensor([F.copy() for F in m.factors]) for m in ms]
    pkg.cp_cals(X, kts, pkg.CalsParams(max_iterations=500, tol=1e-12))
    cc = pkg.core_consistency(X, kts)
    assert all(c > 95 for c, r in zip(cc, ranks) if r <= 3), cc
    assert max(c for c, r in zip(cc, ranks) if r == 5) < min(c for c, r in zip(cc, ranks) if r == 3), cc
    for c, kt in zip(cc, kts):
        assert close(c, corcondia_ref(X, kt.factors, kt.lam))


@pytest.mark.gpu
def test_jackknife_submodels(pkg):
    rng = np.random.default_rng(11)
    X = planted(rng, (12, 15, 14), R=3, noise=0.05)
    ranks = [3] * 6 + [2]
    jk = [(0, i) for i in range(6)] + [(-1, 0)]
    eng = _fit(pkg, X, ranks, seed=5, K=6, jk=jk)
    cc, status = eng.core_consistency()
    fitted = eng.fetch_all()
    _check_against_reference(X, fitted, cc, status, jk)
    for i in range(6):  # the row-deleted problem
        fs, lam, _ = fitted[i]
        Xd = np.delete(X, i, axis=0)
        want = corcondia_ref(Xd, [np.delete(fs[0], i, axis=0)] + list(fs[1:]), lam)
        assert close(cc[i], want), (i, cc[i], want)
    # enqueued without a run: the flagged row is left out as well
    kts = [pkg.Ktensor([F.copy() for F in fs], lam.copy(), *jk[i]) for i, (fs, lam, _) in enumerate(fitted)]
    for k in kts[:6]:
        k.factors[0][k.jk_fiber, :] = 7.0
    got = pkg.core_consistency(X, kts)
    assert np.allclose(got, cc, rtol=1e-10, atol=1e-10)
    eng.close()


@pytest.mark.gpu
def test_queue_longer_than_buffer(pkg):
    rng = np.random.default_rng(2)
    X = planted(rng, (31, 27, 25), R=4, noise=0.5)
    ranks = list(range(1, 21)) * 2
    eng = _fit(pkg, X, ranks, seed=9, K=20, buffer_cols=30, force=False)  # eviction and admission in the run
    small, st_small = eng.core_consistency()  # batches of at most 30 columns
    fitted = eng.fetch_all()
    eng.configure(sum(ranks), 20, 1e-7)
    big, st_big = eng.core_consistency()  # one batch
    assert np.array_equal(small.view(np.int64), big.view(np.int64)) and np.array_equal(st_small, st_big)
    _check_against_reference(X, fitted, big, st_big)
    eng.close()


@pytest.mark.gpu
def test_statuses(pkg):
    rng = np.random.default_rng(4)
    modes = (40, 36, 12)
    X = planted(rng, modes, R=3, noise=0.1)
    good = [[rng.standard_normal((I, r)) for I in modes] for r in (3, 5, 2)]
    r97 = [rng.standard_normal((I, 97)) for I in modes]
    r14 = [rng.standard_normal((I, 14)) for I in modes]  # 14 > 12
    eq = [rng.standard_normal((I, 4)) for I in modes]
    eq[1][:, 2] = eq[1][:, 1]
    queue = [good[0], r97, good[1], r14, eq, good[2]]
    with pkg.Engine(0) as eng:
        eng.set_tensor(X)
        eng.clear_models()
        eng.enqueue_many(queue)
        cc, status = eng.core_consistency()
        eng.clear_models()
        eng.enqueue_many(good)
        cc_good, _ = eng.core_consistency()
    assert list(status) == [0, 1, 0, 2, 2, 0], status
    assert np.isnan(cc[[1, 3, 4]]).all()
    assert np.array_equal(cc[[0, 2, 5]].view(np.int64), cc_good.view(np.int64))
    for c, fs in zip(cc_good, good):
        assert close(c, corcondia_ref(X, fs))
    with pkg.Engine(0) as eng:  # 4 modes: the limit is 64
        X4 = rng.standard_normal((66, 65, 3, 2))
        eng.set_tensor(X4)
        eng.clear_models()
        eng.enqueue_many([[rng.standard_normal((I, 65)) for I in X4.shape]])
        _, st4 = eng.core_consistency()
        assert list(st4) == [1]


@pytest.mark.gpu
def test_refused_tensors(pkg):
    with pkg.Engine(0) as eng:
        eng.set_tensor(np.ones((4, 4, 4, 4, 4)))
        eng.clear_models()
        eng.enqueue_many([[np.ones((4, 1))] * 5])
        with pytest.raises(pkg.CalsB200Error, match="3 and 4 modes"):
            eng.core_consistency()


def _bits(results):
    out = []
    for fs, lam, st in results:
        out += [f.tobytes() for f in fs] + [lam.tobytes(), (st.iters, st.error, st.fit, st.old_fit, st.chol_info)]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("msdt,K", [("1", 3), ("1", 4), ("0", 3)])
def test_no_side_effects(pkg, monkeypatch, msdt, K):
    monkeypatch.setenv("CALS_B200_MSDT", msdt)
    rng = np.random.default_rng(6)
    X = planted(rng, (70, 66, 64), R=4, noise=0.1)
    ranks = [1, 3, 5, 8, 2]
    runs = []
    for call in (False, True):
        eng = _fit(pkg, X, ranks, seed=1, K=K)
        if call:
            eng.core_consistency()
        first = _bits(eng.fetch_all())
        if call:
            eng.core_consistency()
        eng.rerun()
        second = _bits(eng.fetch_all())
        runs.append((first, second))
        eng.close()
    assert runs[0] == runs[1]


CPP_CHECK = r"""
#include <cstdio>
#include <vector>
#include "cals.h"
int main(int argc, char **argv) {
  FILE *f = fopen(argv[1], "rb");
  long long hdr[3];
  if (fread(hdr, 8, 3, f) != 3) return 2;
  const int N = (int)hdr[0], M = (int)hdr[1];
  std::vector<long long> dims(N), ranks(M);
  if (fread(dims.data(), 8, N, f) != (size_t)N || fread(ranks.data(), 8, M, f) != (size_t)M) return 2;
  std::vector<dim_t> modes(dims.begin(), dims.end());
  cals::Tensor X(modes);
  if (fread(X.get_data(), 8, X.get_n_elements(), f) != (size_t)X.get_n_elements()) return 2;
  std::vector<cals::Ktensor> models;
  for (int m = 0; m < M; m++) {
    models.emplace_back((dim_t)ranks[m], modes);
    for (int n = 0; n < N; n++) {
      cals::Matrix &F = models.back().get_factor(n);
      if (fread(F.get_data(), 8, F.get_n_elements(), f) != (size_t)F.get_n_elements()) return 2;
    }
    if (fread(models.back().get_lambda().data(), 8, ranks[m], f) != (size_t)ranks[m]) return 2;
  }
  fclose(f);
  for (double v : cals::core_consistency(X, models, 0))
    printf("%.17g\n", v);
  return 0;
}
"""


@pytest.mark.gpu
def test_cpp_entry_point(pkg):
    rng = np.random.default_rng(8)
    modes = (20, 17, 15)
    X = planted(rng, modes, R=3, noise=0.05)
    ms = caseio.random_models(rng, modes, [1, 3, 4, 6])
    kts = [pkg.Ktensor([F.copy() for F in m.factors]) for m in ms]
    pkg.cp_cals(X, kts, pkg.CalsParams(max_iterations=10, force_max_iter=True))
    want = pkg.core_consistency(X, kts)
    libdir = os.path.join(ROOT, "cp-cals_b200")
    with tempfile.TemporaryDirectory() as tmp:
        src, exe, data = (os.path.join(tmp, n) for n in ("check.cpp", "check", "case.bin"))
        with open(src, "w") as fh:
            fh.write(CPP_CHECK)
        subprocess.run(["g++", "-O1", "-std=c++17", "-I" + os.path.join(ROOT, "include"),
                        "-I" + os.path.join(ROOT, "include", "utils"), "-o", exe, src, "-L" + libdir, "-lcals",
                        "-lcals_b200", "-Wl,-rpath," + libdir], check=True)
        with open(data, "wb") as fh:
            np.array([3, len(kts), 0] + list(modes) + [k.rank for k in kts], dtype=np.int64).tofile(fh)
            np.asfortranarray(X).ravel(order="F").tofile(fh)
            for k in kts:
                for F in k.factors:
                    np.asfortranarray(F).ravel(order="F").tofile(fh)
                k.lam.astype(np.float64).tofile(fh)
        out = subprocess.run([exe, data], capture_output=True, text=True, check=True, timeout=600).stdout.split()
    got = np.array([float(v) for v in out])
    assert np.array_equal(got, want), (got, want)
