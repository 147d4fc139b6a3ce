"""TEST INFRASTRUCTURE -- generates tests/golden/*.npz from the UNMODIFIED reference (oracle/_ref/cals_ref).

Run in the build container (where /root/reference exists and oracle/build_ref.sh has produced oracle/_ref):
    python oracle/make_golden.py
Each fixture stores the seeded inputs (tensor + initial models) and the reference's outputs (factors, lambda, error,
fit_diff, iteration counts, report scalars), so that the oracle and the CUDA path can be checked on machines where the
reference is not present (the GPU box).  The reference ships no golden vectors of its own (SURVEY.md section 4).
The exception is `python oracle/make_golden.py full` (main_full): sampled outputs at BASELINE's full sizes, computed by
the oracle itself, which the fixtures above hold to the reference.
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import caseio  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def lowrank_tensor(rng, modes, rank, noise=0.0):
    fs = [rng.uniform(-1, 1, size=(i, rank)) for i in modes]
    X = caseio.ktensor_to_tensor(fs, np.ones(rank))
    if noise:
        X = X + noise * rng.standard_normal(X.shape)
    return X


def pack(name, X, models, res, **params):
    d = {"X": np.asfortranarray(X), "n_models": len(models), "iter": res.iters, "n_ktensors": res.n_ktensors,
         "comp_sum": res.comp_sum, "x_norm": res.x_norm}
    for k, v in params.items():
        d["param_" + k] = v
    for i, (m_in, m_out) in enumerate(zip(models, res.models)):
        d["m%d_jk" % i] = np.array([m_in.jk_mode, m_in.jk_fiber])
        d["m%d_stats" % i] = np.array([m_out.iters, m_out.error, m_out.fit_diff])
        d["m%d_lam" % i] = m_out.lam
        for n, (fi, fo) in enumerate(zip(m_in.factors, m_out.factors)):
            d["m%d_in%d" % (i, n)] = fi
            d["m%d_out%d" % (i, n)] = fo
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **d)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def main():
    os.makedirs(OUT, exist_ok=True)
    rng = np.random.default_rng(20261018)

    # 1. forced iterations, everything resident, 3 modes (uniform random tensor, like the reference driver)
    modes = (13, 12, 11)
    X = rng.uniform(-1, 1, size=modes)
    ms = caseio.random_models(rng, modes, [1, 2, 3, 4, 5, 6, 7, 8])
    for K in (1, 2, 5):
        p = dict(max_iter=K, tol=1e-7, buffer_size=36, force_max_iter=True)
        pack("forced_3d_k%d" % K, X, ms, caseio.run_reference(X, ms, **p), **p)

    # 2. queueing / eviction / compaction (buffer smaller than the sum of ranks), tol-based, low-rank target
    #    (shape of tests/cals/test_cals.cpp:13-86 SimpleCorrectness, fewer models)
    Xl = lowrank_tensor(rng, modes, 5)
    ranks = list(rng.permutation(np.repeat(np.arange(1, 7), 5)))
    ms = caseio.random_models(rng, modes, ranks)
    p = dict(max_iter=60, tol=1e-5, buffer_size=14, force_max_iter=False)
    pack("queue_tol_3d", Xl, ms, caseio.run_reference(Xl, ms, **p), **p)

    # 3. four modes, odd extents
    modes4 = (5, 7, 4, 6)
    X4 = rng.uniform(-1, 1, size=modes4)
    ms = caseio.random_models(rng, modes4, [1, 3, 2, 5, 4])
    p = dict(max_iter=4, tol=1e-7, buffer_size=9, force_max_iter=True)
    pack("forced_4d_queue", X4, ms, caseio.run_reference(X4, ms, **p), **p)

    # 4. jackknife models mixed with a regular one (shape of tests/cals/test_cals.cpp:181-297 LogicCorrectness)
    modesj = (9, 6, 7)
    Xj = lowrank_tensor(rng, modesj, 3, noise=0.01)
    base = caseio.random_models(rng, modesj, [3])[0]
    ms = []
    for i in range(modesj[0]):
        fs = [F.copy() for F in base.factors]
        fs[0][i, :] = 0.0
        ms.append(caseio.Model(factors=fs, lam=base.lam.copy(), jk_mode=0, jk_fiber=i))
    ms.append(caseio.Model(factors=[F.copy() for F in base.factors], lam=base.lam.copy()))
    p = dict(max_iter=12, tol=1e-4, buffer_size=10, force_max_iter=True)
    pack("jackknife_3d", Xj, ms, caseio.run_reference(Xj, ms, **p), **p)

    # 5. always_evict_first
    ms = caseio.random_models(rng, modes, [2, 3, 1, 4])
    p = dict(max_iter=50, tol=1e-6, buffer_size=10, always_evict_first=True)
    pack("evict_first_3d", X, ms, caseio.run_reference(X, ms, **p), **p)


def main_nnls():
    """Fixtures for update_method == NNLS (reference src/utils/update.cpp:61-176), added after the first set: own
    random stream so that the earlier fixtures stay byte-identical.  `python oracle/make_golden.py nnls`"""
    rng = np.random.default_rng(20261019)
    # non-negative low-rank target + noise, queueing (buffer < sum of ranks), forced iterations
    modes = (14, 12, 10)
    gen = [rng.uniform(0, 1, size=(i, 4)) for i in modes]
    X = caseio.ktensor_to_tensor(gen, np.ones(4)) + 0.02 * rng.standard_normal(modes)
    ms = caseio.random_models(rng, modes, [3, 5, 2, 7, 4, 1])
    p = dict(max_iter=8, tol=1e-7, buffer_size=12, force_max_iter=True, nnls=True)
    pack("nnls_3d_queue", X, ms, caseio.run_reference(X, ms, **p), **p)
    # four modes, tol-based stopping
    modes4 = (6, 5, 4, 7)
    gen = [rng.uniform(0, 1, size=(i, 3)) for i in modes4]
    X4 = caseio.ktensor_to_tensor(gen, np.ones(3)) + 0.01 * rng.standard_normal(modes4)
    ms = caseio.random_models(rng, modes4, [2, 4, 3])
    p = dict(max_iter=30, tol=1e-6, buffer_size=9, force_max_iter=False, nnls=True)
    pack("nnls_4d_tol", X4, ms, caseio.run_reference(X4, ms, **p), **p)


def main_ls():
    """Fixtures for line search (reference src/utils/line_search.cpp), own random stream.
    `python oracle/make_golden.py ls`.  Forced iteration counts on noisy tensors that are still far from converged:
    the accept / go-back decisions compare errors, and on a converged model those differ only in the last bits."""
    rng = np.random.default_rng(20261020)
    modes = (18, 17, 16)
    gen = [rng.uniform(-1, 1, size=(i, 4)) for i in modes]
    X = caseio.ktensor_to_tensor(gen, np.ones(4)) + 0.05 * rng.standard_normal(modes)
    ms = caseio.random_models(rng, modes, [5, 5, 3, 6])
    p = dict(max_iter=14, tol=1e-6, buffer_size=11, force_max_iter=True, line_search=True, ls_method=0, ls_interval=4,
             ls_step=1.2)
    pack("ls_noerr_3d_queue", X, ms, caseio.run_reference(X, ms, **p), **p)
    p = dict(max_iter=13, tol=1e-6, buffer_size=19, force_max_iter=True, line_search=True, ls_method=1, ls_interval=5,
             ls_step=0.0)
    pack("ls_errcheck_3d", X, ms, caseio.run_reference(X, ms, **p), **p)


FULL_SAMPLE_ROWS = 4


def pack_sampled(name, res, seed):
    """Full-size outputs, sampled to stay small: per model one column (seeded choice) of every factor at
    FULL_SAMPLE_ROWS seeded rows per mode, the norm of that whole factor column, its lambda entry, and the model's
    iteration count, error and fit; plus the report scalars."""
    rng = np.random.default_rng(seed)
    N = len(res.models[0].factors)
    rows = [np.sort(rng.choice(F.shape[0], size=min(FULL_SAMPLE_ROWS, F.shape[0]), replace=False))
            for F in res.models[0].factors]
    cols = np.array([int(rng.integers(0, m.rank)) for m in res.models])
    d = {"iter": res.iters, "n_ktensors": res.n_ktensors, "comp_sum": res.comp_sum, "x_norm": res.x_norm, "cols": cols,
         "lam": np.array([m.lam[c] for m, c in zip(res.models, cols)]),
         "iters": np.array([m.iters for m in res.models]), "error": np.array([m.error for m in res.models]),
         "fit": np.array([m.fit for m in res.models])}
    for n in range(N):
        d["rows%d" % n] = rows[n]
        d["f%d" % n] = np.array([m.factors[n][rows[n], c] for m, c in zip(res.models, cols)])
        d["colnorm%d" % n] = np.array([np.linalg.norm(m.factors[n][:, c]) for m, c in zip(res.models, cols)])
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **d)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB", flush=True)


def main_full():
    """Sampled full-size fixtures for tests/test_full_size.py and the bench contract test, computed by the CPU oracle
    (oracle/cals_oracle.c, pinned against the reference's own outputs by tests/test_oracle.py) on the seeded inputs
    those tests build.  `python oracle/make_golden.py full` (about ten minutes on eight cores)."""
    import oracle
    sys.path.insert(0, os.path.dirname(OUT))
    import test_full_size as tfs
    sys.path.insert(0, os.path.dirname(os.path.dirname(OUT)))
    import bench
    for cfg, modes, ranks, seed, Ks in (("config2", (200, 200, 200), [r for r in range(1, 21) for _ in range(10)], 2002,
                                         (1, 2, 3)),
                                        ("config4", (80, 80, 80, 80), [r for r in range(1, 31) for _ in range(5)], 4004,
                                         (1, 2))):
        X, ms = tfs._driver_inputs(modes, ranks, seed)
        for K in Ks:
            res = oracle.cp_cals(X, ms, max_iter=K, force_max_iter=True, buffer_size=sum(ranks))
            pack_sampled("full_%s_k%d" % (cfg, K), res, seed + K)
    X, ms = tfs._config3_inputs()
    res = oracle.cp_cals(X, ms, max_iter=3, force_max_iter=True, buffer_size=sum(m.rank for m in ms))
    pack_sampled("full_config3_jk_k3", res, 3003)
    cfg = bench.CONFIGS[2]
    X, models, jk = bench.workload(cfg, 0)
    ms = [caseio.Model(factors=fs, jk_mode=j[0], jk_fiber=j[1]) for fs, j in zip(models, jk)]
    res = oracle.cp_cals(X, ms, max_iter=cfg["als_iters"], force_max_iter=True, buffer_size=sum(cfg["ranks"]))
    pack_sampled("bench_config2_step", res, 2)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "full":
        main_full()
    elif len(sys.argv) > 1 and sys.argv[1] == "ls":
        main_ls()
    elif len(sys.argv) > 1 and sys.argv[1] == "nnls":
        main_nnls()
    else:
        main()
