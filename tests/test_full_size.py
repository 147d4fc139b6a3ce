"""GPU parity at BASELINE.json's FULL sizes (-m gpu), where the CPU oracle would take minutes: size-independent
properties instead of element-wise comparison of everything.

  * MTTKRP: the tensor-core kernel == the oracle on a random subset of columns (the MTTKRP is column-separable, so a
    column subset of the full-width result must equal the oracle run on just those columns), all modes.
  * cp_cals: the fast error of a fitted model == the explicit ||X - model|| (reference tests/als/test_als.cpp:125-145),
    a model fitted among 200 concurrent ones == the same model fitted alone (reference tests/cals/test_cals.cpp:13-86),
    the error never increases from one ALS iteration to the next.
  * jackknife (config 3 shape): a flagged model == ALS on the row-deleted tensor (reference tests/cals/test_cals.cpp:181-297).
"""
import os

import numpy as np
import pytest

import caseio
import oracle
from helpers import RTOL, assert_models_close, assert_sampled_models_close, load_sampled, rel_err, to_ktensors

pytestmark = pytest.mark.gpu


def _driver_inputs(modes, ranks, seed):
    """Inputs as the reference driver makes them (src/examples/driver.cpp:133-153): X uniform(-1,1), models uniform(-1,1)
    then Ktensor::normalize()."""
    rng = np.random.default_rng(seed)
    X = np.asfortranarray(rng.uniform(-1.0, 1.0, size=modes))
    return X, caseio.random_models(rng, modes, ranks)


def _config3_inputs():
    """BASELINE config 3 shape (299 x 301 x 41): all 299 leave-one-out sub-models of one rank-5 base model."""
    rng = np.random.default_rng(3003)
    modes, R = (299, 301, 41), 5
    gen = [rng.uniform(0, 1, size=(i, R)) for i in modes]
    X = np.asfortranarray(caseio.ktensor_to_tensor(gen, np.ones(R)) + 0.01 * rng.standard_normal(modes))
    base = caseio.random_models(rng, modes, [R])[0]
    ms = []
    for i in range(modes[0]):
        fs = [F.copy() for F in base.factors]
        fs[0][i, :] = 0.0  # Ktensor::set_jk_fiber(0.0) as jk_cp_cals leaves its inputs (src/utils/utils.cpp:40-51)
        ms.append(caseio.Model(factors=fs, lam=base.lam.copy(), jk_mode=0, jk_fiber=i))
    return X, ms


def _against_stored(pkg, eng, X, ms, K, name, what, methods=("auto", "mttkrp")):
    """The same clause against stored full-size outputs (tests/golden/<name>.npz, oracle/make_golden.py full): the CPU
    oracle, which tests/test_oracle.py holds to the reference's own outputs, sampled per model (see
    assert_sampled_models_close).  Runs everywhere; the live comparison with the reference below runs where a build of
    the reference exists."""
    C = sum(m.rank for m in ms)
    want = load_sampled(name)
    for method in methods:
        kts = to_ktensors(pkg, ms)
        rep = pkg.cp_cals(X, kts, pkg.CalsParams(max_iterations=K, buffer_size=C, force_max_iter=True,
                                                 mttkrp_method=method), engine=eng)
        assert (rep.iter, rep.n_ktensors, rep.ktensor_comp_sum) == (want["iter"], want["n_ktensors"], want["comp_sum"])
        assert abs(rep.X_norm - want["x_norm"]) <= 1e-12 * want["x_norm"]
        assert_sampled_models_close(kts, want, rtol=RTOL, what="%s K=%d %s:" % (what, K, method))


def _against_reference(pkg, eng, X, ms, K, what, methods=("auto", "mttkrp")):
    """north_star's correctness clause at full size: from identical initial factors, after a fixed iteration count, every
    factor matrix, lambda and fit within 1e-9 of the UNMODIFIED reference's CPU cals::cp_cals (pattern:
    reference tests/cals/test_cals.cpp:13-86).  Both mttkrp_method settings of this path (pair nodes / one MTTKRP per
    mode) are held to it."""
    C = sum(m.rank for m in ms)
    if not caseio.ref_available():
        return None
    ref = caseio.run_reference(X, ms, max_iter=K, force_max_iter=True, buffer_size=C, threads=os.cpu_count() or 1)
    assert ref.iters == K and ref.n_ktensors == len(ms)
    worst = 0.0
    for method in methods:
        kts = to_ktensors(pkg, ms)
        rep = pkg.cp_cals(X, kts, pkg.CalsParams(max_iterations=K, buffer_size=C, force_max_iter=True,
                                                 mttkrp_method=method), engine=eng)
        assert (rep.iter, rep.n_ktensors, rep.ktensor_comp_sum) == (ref.iters, ref.n_ktensors, ref.comp_sum)
        assert rep.pair_node == (method != "mttkrp" and X.ndim in (3, 4))
        assert abs(rep.X_norm - ref.x_norm) <= 1e-12 * ref.x_norm
        assert_models_close(kts, ref.models, ref.x_norm, rtol=RTOL, what="%s K=%d %s:" % (what, K, method))
        for g, r in zip(kts, ref.models):  # fit = 1 - |err| / ||X|| (include/ktensor.h:178-183), per model
            assert abs(g.fit - (1.0 - abs(r.error) / ref.x_norm)) <= RTOL
            assert abs(g.fit_diff - r.fit_diff) <= RTOL
            worst = max(worst, max(rel_err(a, b) for a, b in zip(g.factors, r.factors)))
    return worst


@pytest.mark.parametrize("K", [1, 2, 3])
def test_config2_all_models_vs_reference(pkg, K):
    """BASELINE config 2 in full -- 200^3 tensor, all 200 models (ranks 1..20 x10), buffer 2100 -- after K = 1, 2, 3
    forced ALS iterations (i.e. per iteration) against the stored outputs and, where built, the unmodified reference."""
    X, ms = _driver_inputs((200, 200, 200), [r for r in range(1, 21) for _ in range(10)], 2002)
    with pkg.Engine(0) as eng:
        _against_stored(pkg, eng, X, ms, K, "full_config2_k%d" % K, "config 2")
        worst = _against_reference(pkg, eng, X, ms, K, "config 2")
    if worst is not None:
        print("config 2, K=%d: worst factor rel err vs reference %.2e" % (K, worst))


@pytest.mark.parametrize("K", [1, 2])
def test_config4_all_models_vs_reference(pkg, K):
    """BASELINE config 4 in full -- 80^4 tensor, 150 models (ranks 1..30 x5), buffer 2325.  The reference materialises
    its 9.5 GB Khatri-Rao workspace for this (src/cals.cpp:78-88)."""
    X, ms = _driver_inputs((80, 80, 80, 80), [r for r in range(1, 31) for _ in range(5)], 4004)
    with pkg.Engine(0) as eng:
        _against_stored(pkg, eng, X, ms, K, "full_config4_k%d" % K, "config 4")
        worst = _against_reference(pkg, eng, X, ms, K, "config 4")
    if worst is not None:
        print("config 4, K=%d: worst factor rel err vs reference %.2e" % (K, worst))


def test_config3_all_submodels_vs_reference(pkg):
    """BASELINE config 3 shape (299 x 301 x 41): all 299 leave-one-out sub-models of one rank-5 base model, K = 3, against
    the jackknife branches (reference src/cals.cpp:198-200 norms, :250-251 zeroed fibre, :291-293 error)."""
    X, ms = _config3_inputs()
    K = 3
    with pkg.Engine(0) as eng:
        _against_stored(pkg, eng, X, ms, K, "full_config3_jk_k3", "config 3 jackknife")
        worst = _against_reference(pkg, eng, X, ms, K, "config 3 jackknife")
    if worst is not None:
        print("config 3, %d sub-models, K=%d: worst factor rel err vs reference %.2e" % (len(ms), K, worst))


def _subset_check(pkg, eng, X, fs, n_check, rng, tol=1e-11):
    C = fs[0].shape[1]
    cols = np.sort(rng.choice(C, size=n_check, replace=False))
    sub = [np.asfortranarray(F[:, cols]) for F in fs]
    for n in range(X.ndim):
        got, ms = eng.mttkrp(fs, n)
        want = oracle.mttkrp(X, sub, n)
        ce = np.linalg.norm(got[:, cols] - want, axis=0) / np.linalg.norm(want, axis=0)
        assert ce.max() <= tol, "mode %d worst checked column %.3e" % (n, ce.max())
        assert np.isfinite(got).all()


def test_config2_mttkrp_full_width(pkg):
    rng = np.random.default_rng(202)
    modes, C = (200, 200, 200), 2100
    X = rng.uniform(-1, 1, size=modes)
    fs = [np.asfortranarray(rng.uniform(-1, 1, size=(i, C))) for i in modes]
    with pkg.Engine(0) as eng:
        eng.set_tensor(X)
        _subset_check(pkg, eng, X, fs, 12, rng)
        # linearity in one factor: MTTKRP(.., 2*A_1 + B_1, ..) = 2*MTTKRP(.., A_1, ..) + MTTKRP(.., B_1, ..)
        B1 = np.asfortranarray(rng.uniform(-1, 1, size=(modes[1], C)))
        g_a, _ = eng.mttkrp(fs, 0)
        g_b, _ = eng.mttkrp([fs[0], B1, fs[2]], 0)
        g_ab, _ = eng.mttkrp([fs[0], np.asfortranarray(2 * fs[1] + B1), fs[2]], 0)
        assert rel_err(g_ab, 2 * g_a + g_b) <= 1e-12


def test_config4_mttkrp_full_width(pkg):
    rng = np.random.default_rng(404)
    modes, C = (80, 80, 80, 80), 2325
    X = rng.uniform(-1, 1, size=modes)
    fs = [np.asfortranarray(rng.uniform(-1, 1, size=(i, C))) for i in modes]
    with pkg.Engine(0) as eng:
        eng.set_tensor(X)
        _subset_check(pkg, eng, X, fs, 6, rng)


def _explicit_error(X, kt):
    N = X.ndim
    letters = "abcdefgh"[:N]
    expr = ",".join(l + "r" for l in letters) + ",r->" + letters
    M = np.einsum(expr, *kt.factors, kt.lam, optimize=True)
    return float(np.linalg.norm(X - M))


@pytest.mark.parametrize("modes,ranks,K", [
    ((200, 200, 200), [r for r in range(1, 21) for _ in range(10)], 3),   # config 2
    ((80, 80, 80, 80), [r for r in range(1, 31) for _ in range(5)], 2),   # config 4
])
def test_full_config_cp_cals_properties(pkg, modes, ranks, K):
    rng = np.random.default_rng(len(modes))
    # low-rank + noise so that the fits are non-trivial and differ between models
    gen = [rng.uniform(-1, 1, size=(i, 6)) for i in modes]
    X = caseio.ktensor_to_tensor(gen, np.ones(6)) + 0.05 * rng.standard_normal(modes)
    ms = caseio.random_models(rng, modes, ranks)
    C = sum(ranks)
    probe = [0, len(ranks) // 2, len(ranks) - 1]  # smallest, middle and largest rank
    with pkg.Engine(0) as eng:
        prev_err = None
        for k in (K - 1, K):
            kts = to_ktensors(pkg, ms)
            rep = pkg.cp_cals(X, kts, pkg.CalsParams(max_iterations=k, buffer_size=C, force_max_iter=True), engine=eng)
            assert rep.iter == k and rep.n_ktensors == len(ranks) and rep.ktensor_comp_sum == C
            err = np.array([kt.error for kt in kts])
            if prev_err is not None:  # ALS never increases the error
                assert (err <= prev_err * (1 + 1e-9)).all()
            prev_err = err
        xn = rep.X_norm
        assert abs(xn - np.linalg.norm(X)) <= 1e-12 * xn
        # pair nodes (default, csrc/pairnode.cuh) == one full MTTKRP per mode, at full size
        assert rep.pair_node
        per_mode = to_ktensors(pkg, ms)
        rep1 = pkg.cp_cals(X, per_mode, pkg.CalsParams(max_iterations=K, buffer_size=C, force_max_iter=True,
                                                        mttkrp_method="mttkrp"), engine=eng)
        assert not rep1.pair_node
        assert max(abs(a.fit - b.fit) for a, b in zip(kts, per_mode)) <= 1e-10
        for i in probe:
            for Fa, Fb in zip(kts[i].factors, per_mode[i].factors):
                assert rel_err(Fa, Fb) <= RTOL
        for i in probe:
            kt = kts[i]
            # fast error == explicit error, fit consistent
            assert abs(kt.error - _explicit_error(X, kt)) <= 1e-9 * xn
            assert abs(kt.fit - (1 - kt.error / xn)) <= 1e-13
            # concurrent == alone
            alone = to_ktensors(pkg, [ms[i]])
            pkg.cp_cals(X, alone, pkg.CalsParams(max_iterations=K, buffer_size=ranks[i], force_max_iter=True),
                        engine=eng)
            for Fa, Fc in zip(alone[0].factors, kt.factors):
                assert rel_err(Fc, Fa) <= RTOL
            assert rel_err(kt.lam, alone[0].lam) <= RTOL and abs(kt.fit - alone[0].fit) <= RTOL


def test_config3_jackknife_equals_row_deleted_als(pkg):
    rng = np.random.default_rng(3)
    modes, R = (299, 301, 41), 5
    gen = [rng.uniform(0, 1, size=(i, R)) for i in modes]
    X = caseio.ktensor_to_tensor(gen, np.ones(R)) + 0.01 * rng.standard_normal(modes)
    base = caseio.random_models(rng, modes, [R])[0]
    fibers = [0, 150, 298]
    K = 5
    with pkg.Engine(0) as eng:
        flagged = [pkg.Ktensor([F.copy() for F in base.factors], None, 0, f) for f in fibers]
        for kt in flagged:
            kt.set_jk_fiber(0.0)
        rep = pkg.cp_cals(X, flagged, pkg.CalsParams(max_iterations=K, buffer_size=3 * R, force_max_iter=True),
                          engine=eng)
        assert rep.iter == K
        jkn = eng.jk_norms()
        for kt, f in zip(flagged, fibers):
            Xd = np.delete(X, f, axis=0)
            assert abs(jkn[f] - np.linalg.norm(Xd)) <= 1e-11 * rep.X_norm
            alone = pkg.Ktensor([np.delete(base.factors[0], f, axis=0)] + [F.copy() for F in base.factors[1:]])
            pkg.cp_cals(Xd, [alone], pkg.CalsParams(max_iterations=K, buffer_size=R, force_max_iter=True), engine=eng)
            got0 = np.delete(kt.factors[0], f, axis=0)
            assert np.all(kt.factors[0][f] == 0.0)
            assert rel_err(got0, alone.factors[0]) <= RTOL
            for n in (1, 2):
                assert rel_err(kt.factors[n], alone.factors[n]) <= RTOL
            assert rel_err(kt.lam, alone.lam) <= RTOL
            assert abs(kt.error - alone.error) <= RTOL * rep.X_norm


def test_edge_cases(pkg):
    rng = np.random.default_rng(9)
    with pkg.Engine(0) as eng:
        X = rng.uniform(-1, 1, size=(6, 5, 4))
        # empty queue and a model that can never be admitted are refused with a message, not a hang
        with pytest.raises(pkg.CalsB200Error):
            pkg.cp_cals(X, [], pkg.CalsParams(max_iterations=2, buffer_size=4), engine=eng)
        with pytest.raises(pkg.CalsB200Error):
            pkg.cp_cals(X, to_ktensors(pkg, caseio.random_models(rng, X.shape, [5])),
                        pkg.CalsParams(max_iterations=2, buffer_size=4), engine=eng)
        # a single rank-1 model (C = 1), a mode of extent 1, and a rank larger than every extent
        for modes, ranks in [((6, 5, 4), [1]), ((6, 1, 5), [2, 1]), ((3, 4, 2), [7])]:
            X = rng.uniform(-1, 1, size=modes)
            ms = caseio.random_models(rng, modes, ranks)
            want = oracle.cp_cals(X, ms, max_iter=3, force_max_iter=True)
            kts = to_ktensors(pkg, ms)
            pkg.cp_cals(X, kts, pkg.CalsParams(max_iterations=3, buffer_size=sum(ranks), force_max_iter=True),
                        engine=eng)
            for g, w in zip(kts, want.models):
                if g.chol_info or w.chol_fail:  # rank > extents: the Hadamard of Grams is singular, nothing to compare
                    assert bool(g.chol_info) == bool(w.chol_fail)
                    continue
                for Fg, Fw in zip(g.factors, w.factors):
                    assert rel_err(Fg, Fw) <= 1e-7
                assert abs(g.fit - w.fit) <= 1e-7


@pytest.mark.skipif(not __import__("os").environ.get("CALS_B200_BIG"), reason="opt-in (CALS_B200_BIG=1): 8 GB tensor, "
                    "about two minutes of host time for the generation and the CPU oracle")
def test_config5_mttkrp_full_size(pkg):
    """BASELINE config 5 at full size on ONE GPU: 1000^3 tensor (8 GB; byte offsets beyond 2^32), C = 1275 columns.
    The tensor-core MTTKRP of every mode against the CPU oracle on a few columns, and the slab formulation (tensor cut
    in two along the last mode, partial results added on the host) against the unsliced one on all columns."""
    import importlib
    d = importlib.import_module("cp_cals_b200.distributed")
    rng = np.random.default_rng(5)
    modes, C = (1000, 1000, 1000), 1275
    X = np.empty(modes, order="F")
    flat = X.reshape(-1, order="F")
    for o in range(0, flat.size, 1 << 24):
        flat[o:o + (1 << 24)] = rng.uniform(-1, 1, size=min(1 << 24, flat.size - o))
    fs = [np.asfortranarray(rng.uniform(-1, 1, size=(i, C))) for i in modes]
    cols = np.sort(rng.choice(C, size=3, replace=False))
    sub = [np.asfortranarray(F[:, cols]) for F in fs]
    full = []
    with pkg.Engine(0) as eng:
        eng.set_tensor(X)
        assert abs(eng.tensor_norm() - np.sqrt(np.sum(np.square(flat)))) <= 1e-10 * eng.tensor_norm()
        for n in range(3):
            got, ms = eng.mttkrp(fs, n, repeats=2)
            want = oracle.mttkrp(X, sub, n)
            ce = np.linalg.norm(got[:, cols] - want, axis=0) / np.linalg.norm(want, axis=0)
            assert ce.max() <= 1e-11, "mode %d worst checked column %.3e" % (n, ce.max())
            full.append(got)
            print("mode %d: %.2f ms, %.1f TFLOP/s" % (n, ms, 2.0 * X.size * C / ms / 1e9))
    cuts = [0] + [hi for _, hi in d.shard_slabs(modes[2], 2)]
    acc = [np.zeros_like(g) for g in full]
    for r in range(2):
        with pkg.Engine(0) as eng:
            eng.comm_alloc(r, 2, d.exchange_capacity(modes, C))
            eng.set_tensor_slab(modes, 2, cuts, X[:, :, cuts[r]:cuts[r + 1]])
            for n in range(3):
                part, _ = eng.mttkrp(fs, n)
                acc[n] += part
    for n in range(3):
        assert rel_err(acc[n], full[n]) <= 1e-12
