"""Launch paths, tuning knobs and state kept between calls (csrc/engine.cu: run_loop, prepare_run, install_tensor).

The parity suite runs the default launch path: the replayed CUDA graph with the default knobs.  run_loop has other host
sequences that enqueue the same iteration -- the timed graph (and, with line search, plain launches with events), the
no-graph path with host run-ahead, other graph batch sizes, programmatic dependent launch, the forked prefactor branch --
and knobs that change the arithmetic (fused partial-tile reduction, narrow column tail, tile height).  This file runs
every workload below on every such path and compares:

- the default path with the oracle (RTOL);
- paths that only change how the same kernels are launched with the default path, bit for bit (every reduction has a
  fixed order, so a difference is a race, a missing launch or a stale buffer);
- paths that change the arithmetic with the default path (1e-11) and the oracle (RTOL);
- the discrete outcomes (iterations, admissions, columns per pass, contractions) on every path;
- that each knob took effect (launch counts derived from enqueue_iteration, kernel names, stderr).

Most knobs are `static const` in the library and read once per process, so every knob setting runs in a subprocess:
`python tests/test_launch_paths.py --worker CASES.npz OUT.npz` fits the cases of CASES.npz and writes the results.

The second part runs a sequence of calls in one Engine -- new tensor contents at the same shape, alternating settings,
changing rank sequences, rerun() -- and requires each result to be bit-identical to the same call on a fresh Engine.
"""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if __name__ == "__main__":  # worker: the same import paths as tests/conftest.py
    for p in (os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), ROOT):
        sys.path.insert(0, p)

import caseio  # noqa: E402
from helpers import RTOL, assert_models_close, rel_err, to_ktensors  # noqa: E402

pytestmark = pytest.mark.gpu

WORKER_TIMEOUT = 900  # seconds per knob setting; the whole matrix of one setting takes a few seconds on a B200
STATS = ("iters", "error", "fit", "old_fit", "chol_info")
REPORT = ("iter", "n_ktensors", "ktensor_comp_sum", "tensor_flops", "sweep_period", "kernel_launches", "X_norm",
          "device_ms", "mttkrp_ms", "update_ms", "pair_node")


# ---------------------------------------------------------------------------------------------------------------------
# workloads
def _workloads():
    """name -> (X, models, CalsParams keyword arguments).  Each one is there for a path it reaches."""
    W = {}

    # A: MSDT-eligible (every extent >= 64), ragged ranks, one jackknife model, forced K = 5 with the whole queue
    #    resident: both parities, the batch graphs and the known_passes stop.
    rng = np.random.default_rng(101)
    modes = (72, 66, 64)
    X = rng.uniform(-1, 1, size=modes)
    ms = caseio.random_models(rng, modes, [3, 7, 1, 12, 5, 9, 2])
    ms[1].jk_mode, ms[1].jk_fiber = 0, 5
    W["A"] = (X, ms, dict(max_iterations=5, buffer_size=39, force_max_iter=True))
    # B: the same with a buffer smaller than the queue: odd passes that move columns fall back to mode 0's own MTTKRP,
    #    and the pass count is not known in advance (run-ahead, `done` flag).
    W["B"] = (X, ms, dict(max_iterations=5, buffer_size=14, force_max_iter=True))

    # C: one-sweep pair node (the 31-long mode keeps MSDT off), 263 columns = ragged last octet and a 7-column narrow
    #    tail, a 299-row mode for which the height rule picks 7.
    rng = np.random.default_rng(102)
    modes = (299, 31, 41)
    X = rng.uniform(-1, 1, size=modes)
    W["C"] = (X, caseio.random_models(rng, modes, [20] * 13 + [3]), dict(max_iterations=3, buffer_size=263,
                                                                        force_max_iter=True))

    # D: 4 modes (two pair nodes, the Xq layout), 360 columns.
    rng = np.random.default_rng(103)
    modes = (20, 44, 9, 31)
    X = rng.uniform(-1, 1, size=modes)
    W["D"] = (X, caseio.random_models(rng, modes, [24] * 15), dict(max_iterations=3, buffer_size=360,
                                                                  force_max_iter=True))

    # E: one MTTKRP per mode, 75 columns (an 11-column narrow tail); the only place FUSED_REDUCE acts on every mode.
    #    Row counts 64 / 48 / 23: the height rule picks tiles of 4 / 6 / 4 row groups, WM_MAX=8 gives 8 / 6 / 4.
    rng = np.random.default_rng(104)
    modes = (64, 48, 23)
    X = rng.uniform(-1, 1, size=modes)
    W["E"] = (X, caseio.random_models(rng, modes, [10, 20, 30, 15]),
              dict(max_iterations=4, buffer_size=75, force_max_iter=True, mttkrp_method="mttkrp"))

    # F: wide (130, 97) and narrow models together on an MSDT-eligible shape, whole queue and queueing.
    rng = np.random.default_rng(105)
    modes = (66, 64, 70)
    XF = rng.uniform(-1, 1, size=modes)
    msF = caseio.random_models(rng, modes, [130, 7, 97, 20])
    W["F1"] = (XF, msF, dict(max_iterations=3, buffer_size=254, force_max_iter=True))
    W["F2"] = (XF, msF, dict(max_iterations=3, buffer_size=140, force_max_iter=True))

    # G: NNLS with queueing.
    rng = np.random.default_rng(106)
    modes = (40, 36, 34)
    gen = [rng.uniform(0, 1, size=(i, 3)) for i in modes]
    X = caseio.ktensor_to_tensor(gen, np.ones(3)) + 0.05 * rng.uniform(0, 1, size=modes)
    W["G"] = (X, caseio.random_models(rng, modes, [3, 5, 4, 2, 6]),
              dict(max_iterations=6, buffer_size=12, force_max_iter=True, update_method="nnls"))

    # H: line search, both methods (with timing on, plain stream launches with events instead of the timed graph).
    rng = np.random.default_rng(107)
    modes = (30, 28, 26)
    gen = [rng.uniform(0, 1, size=(i, 3)) for i in modes]
    X = caseio.ktensor_to_tensor(gen, np.ones(3)) + 0.02 * rng.standard_normal(modes)
    ms = caseio.random_models(rng, modes, [3, 4, 2, 5, 3])
    for name, method in (("H0", "no-error-checking"), ("H1", "error-checking-serial")):
        W[name] = (X, ms, dict(max_iterations=8, buffer_size=10, force_max_iter=True, line_search=True,
                               line_search_interval=3, line_search_method=method))

    # I: unforced stopping on tol with queueing: run-ahead and the `done` flag end the loop.
    rng = np.random.default_rng(108)
    modes = (30, 28, 26)
    gen = [rng.uniform(0, 1, size=(i, 3)) for i in modes]
    X = caseio.ktensor_to_tensor(gen, np.ones(3)) + 0.01 * rng.standard_normal(modes)
    W["I"] = (X, caseio.random_models(rng, modes, [1, 2, 3, 4, 2, 3, 1, 5]),
              dict(max_iterations=60, tol=1e-5, buffer_size=9))

    # T130 / T20: the update window of the timed path with one wide model against one narrow model (F's shape)
    W["T130"] = (XF, [msF[0]], dict(max_iterations=5, buffer_size=130, force_max_iter=True))
    W["T20"] = (XF, [msF[3]], dict(max_iterations=5, buffer_size=130, force_max_iter=True))
    return W


MATRIX = ["A", "B", "C", "D", "E", "F1", "F2", "G", "H0", "H1", "I"]
LENIENT = {"I"}  # tol stopping can flip by one iteration through rounding (test_cp_cals_queue_tol_golden)

# knob setting -> (environment, timing levels run in that process)
SETTINGS = {
    "default": ({}, (0, 1)),
    "no_graph": ({"CALS_B200_NO_GRAPH": "1"}, (0, 1)),
    "graph_batch_1": ({"CALS_B200_GRAPH_BATCH": "1"}, (0,)),
    "graph_batch_4": ({"CALS_B200_GRAPH_BATCH": "4"}, (0,)),
    "graph_batch_64": ({"CALS_B200_GRAPH_BATCH": "64"}, (0,)),
    "pdl": ({"CALS_B200_PDL": "1"}, (0,)),
    "prefactor": ({"CALS_B200_PREFACTOR": "1"}, (0,)),
    "pdl_prefactor": ({"CALS_B200_PDL": "1", "CALS_B200_PREFACTOR": "1"}, (0,)),
    "update_prof": ({"CALS_B200_UPDATE_PROF": "1"}, (0,)),
    "fused_reduce": ({"CALS_B200_FUSED_REDUCE": "1"}, (0,)),
    "narrow": ({"CALS_B200_NARROW": "1"}, (0,)),
    "wm_max_4": ({"CALS_B200_WM_MAX": "4"}, (0,)),
    "wm_max_8": ({"CALS_B200_WM_MAX": "8"}, (0,)),
}
# same kernels, same reduction splits: bit-identical to the default path.  The prefactor branch moves H, its Cholesky
# factor and the block inverses into a kernel of their own, with the same operations in the same order: bit-identical too
# (measured on every workload it runs on).
BITWISE = {"default+timing", "no_graph", "no_graph+timing", "graph_batch_1", "graph_batch_4", "graph_batch_64", "pdl",
           "update_prof", "prefactor", "pdl_prefactor"}
# other arithmetic (tile heights, where the partial tiles are summed): within 1e-11
CLOSE = {"fused_reduce", "narrow", "wm_max_4", "wm_max_8"}
PATHS = ["default+timing", "no_graph", "no_graph+timing", "graph_batch_1", "graph_batch_4", "graph_batch_64", "pdl",
         "prefactor", "pdl_prefactor", "update_prof", "fused_reduce", "narrow", "wm_max_4", "wm_max_8"]
# combinations the engine gates off by design: the knob does nothing there, the run would repeat the default one
SKIP = {
    ("G", "prefactor"): "NNLS: the prefactor branch is off (the active-set solve needs the whole update)",
    ("G", "pdl_prefactor"): "NNLS: the prefactor branch is off",
    ("H0", "prefactor"): "line search: the prefactor branch is off", ("H1", "prefactor"): "line search: prefactor off",
    ("H0", "pdl_prefactor"): "line search: PDL and prefactor are off", ("H1", "pdl_prefactor"): "line search: both off",
    ("H0", "pdl"): "line search: PDL is off", ("H1", "pdl"): "line search: PDL is off",
    ("F1", "fused_reduce"): "a wide model reads G: the separate reduce always runs",
    ("F2", "fused_reduce"): "a wide model reads G: the separate reduce always runs",
}
# knob settings that switch the multi-sweep schedule off by design: NARROW (the narrow instance's tiles carry no
# fused-leaf partials) and FUSED_REDUCE (mode 0 would sum stream-K partials its pair leaf never wrote)
SCHEDULE_OFF = {("A", "narrow"), ("B", "narrow"), ("F1", "narrow"), ("F2", "narrow"), ("A", "fused_reduce"),
                ("B", "fused_reduce")}
# runs recorded with torch.profiler (kernel and runtime-call names)
PROFILED = {"default": ["C", "E"], "no_graph": ["E"], "narrow": ["C", "E"], "wm_max_4": ["E"], "wm_max_8": ["E"]}


def _setting_of(path):
    return path.split("+")[0]


def _runs_for(setting):
    env, timings = SETTINGS[setting]
    runs = []
    for t in timings:
        path = setting if t == 0 else setting + "+timing"
        for w in MATRIX:
            if (w, setting) not in SKIP:
                runs.append(dict(tag="%s|%s" % (w, path), workload=w, timing=t, profile=False))
    if setting == "default":
        runs += [dict(tag="%s|timing" % w, workload=w, timing=1, profile=False) for w in ("T130", "T20")]
    runs += [dict(tag="%s|profile" % w, workload=w, timing=0, profile=True) for w in PROFILED.get(setting, [])]
    return runs


# ---------------------------------------------------------------------------------------------------------------------
# worker side
def _pack_cases(path, runs):
    W = _workloads()
    used = sorted({r["workload"] for r in runs})
    arrays, meta = {}, {}
    for w in used:
        X, ms, params = W[w]
        arrays["%s_X" % w] = np.asfortranarray(X)
        for i, m in enumerate(ms):
            for n, F in enumerate(m.factors):
                arrays["%s_m%d_f%d" % (w, i, n)] = np.asfortranarray(F)
        arrays["%s_jk" % w] = np.array([[m.jk_mode, m.jk_fiber] for m in ms], dtype=np.int64)
        meta[w] = dict(params=params, n_models=len(ms))
    np.savez(path, spec=np.array(json.dumps(dict(runs=runs, workloads=meta))), **arrays)


def _unpack_workload(d, meta, w):
    X = d["%s_X" % w]
    jk = d["%s_jk" % w]
    ms = [caseio.Model(factors=[d["%s_m%d_f%d" % (w, i, n)] for n in range(X.ndim)], jk_mode=int(jk[i, 0]),
                       jk_fiber=int(jk[i, 1])) for i in range(meta[w]["n_models"])]
    return X, ms, meta[w]["params"]


def _worker(cases_path, out_path):
    from conftest import load_package
    pkg = load_package()
    d = np.load(cases_path)
    spec = json.loads(str(d["spec"]))
    out, reports = {}, []
    for k, run in enumerate(spec["runs"]):
        X, ms, params = _unpack_workload(d, spec["workloads"], run["workload"])
        kts = to_ktensors(pkg, ms)
        names = None
        with pkg.Engine(0) as eng:
            if run["profile"]:
                import torch
                from torch.profiler import ProfilerActivity, profile
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    rep = pkg.cp_cals(X, kts, pkg.CalsParams(**params), engine=eng, timing=run["timing"])
                    torch.cuda.synchronize()
                names = sorted({e.name for e in prof.events()})
            else:
                rep = pkg.cp_cals(X, kts, pkg.CalsParams(**params), engine=eng, timing=run["timing"])
            cols = eng.iteration_cols()
        r = {f: getattr(rep, f) for f in REPORT}
        r["pair_node"] = bool(r["pair_node"])
        r["tag"], r["kernels"] = run["tag"], names
        reports.append(r)
        out["r%d_cols" % k] = cols
        out["r%d_stats" % k] = np.array([[float(getattr(kt, s)) for s in STATS] for kt in kts])
        for i, kt in enumerate(kts):
            out["r%d_m%d_lam" % (k, i)] = kt.lam
            for n, F in enumerate(kt.factors):
                out["r%d_m%d_f%d" % (k, i, n)] = F
    np.savez(out_path, reports=np.array(json.dumps(reports)), **out)


class _Fit:
    """One model's result as the helpers of tests/helpers.py expect it."""

    def __init__(self, factors, lam, stats):
        self.factors, self.lam = factors, lam
        self.iters, self.error, self.fit, self.old_fit, self.chol_info = (int(stats[0]), stats[1], stats[2], stats[3],
                                                                         int(stats[4]))


class _Run:
    def __init__(self, d, k, report, n_modes):
        self.report = report
        self.cols = d["r%d_cols" % k]
        st = d["r%d_stats" % k]
        self.models = [_Fit([d["r%d_m%d_f%d" % (k, i, n)] for n in range(n_modes)], d["r%d_m%d_lam" % (k, i)], st[i])
                       for i in range(len(st))]


# ---------------------------------------------------------------------------------------------------------------------
# parent side
@pytest.fixture(scope="module")
def workloads():
    return _workloads()


@pytest.fixture(scope="module")
def oracle_results(workloads):
    import oracle
    cache = {}

    def get(w):
        if w not in cache:
            X, ms, p = workloads[w]
            cache[w] = oracle.cp_cals(X, ms, max_iter=p["max_iterations"], tol=p.get("tol", 1e-7),
                                      buffer_size=p["buffer_size"], force_max_iter=p.get("force_max_iter", False),
                                      nnls=p.get("update_method") == "nnls", line_search=p.get("line_search", False),
                                      ls_method=1 if p.get("line_search_method") == "error-checking-serial" else 0,
                                      ls_interval=p.get("line_search_interval", 5))
        return cache[w]
    return get


@pytest.fixture(scope="module")
def setting_results(tmp_path_factory, workloads):
    """knob setting -> ({tag: _Run}, stderr of the worker); each setting's worker runs once per module."""
    cache = {}

    def get(setting):
        if setting not in cache:
            d = tmp_path_factory.mktemp("worker_" + setting)
            runs = _runs_for(setting)
            _pack_cases(str(d / "cases.npz"), runs)
            env = {k: v for k, v in os.environ.items() if not k.startswith("CALS_B200_")}
            env.update(SETTINGS[setting][0])
            proc = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", str(d / "cases.npz"),
                                   str(d / "out.npz")], env=env, cwd=str(d), capture_output=True, text=True,
                                  timeout=WORKER_TIMEOUT)
            assert proc.returncode == 0, "worker %s failed:\n%s\n%s" % (setting, proc.stdout[-4000:],
                                                                       proc.stderr[-4000:])
            o = np.load(str(d / "out.npz"))
            reports = json.loads(str(o["reports"]))
            res = {}
            for k, r in enumerate(reports):
                w = r["tag"].split("|")[0]
                res[r["tag"]] = _Run(o, k, r, workloads[w][0].ndim)
            cache[setting] = (res, proc.stderr)
        return cache[setting]
    return get


def _result(setting_results, w, path):
    return setting_results(_setting_of(path))[0]["%s|%s" % (w, path)]


def _assert_close_or_equal(got, ref, bitwise, tol, what):
    for i, (g, r) in enumerate(zip(got.models, ref.models)):
        tag = "%s model %d" % (what, i)
        assert g.iters == r.iters, tag + ": iters %d != %d" % (g.iters, r.iters)
        if bitwise:
            for n, (Fg, Fr) in enumerate(zip(g.factors, r.factors)):
                assert np.array_equal(Fg, Fr), tag + ": factor %d differs, rel %.3e" % (n, rel_err(Fg, Fr))
            assert np.array_equal(g.lam, r.lam), tag + ": lambda differs"
            assert (g.error, g.fit, g.old_fit, g.chol_info) == (r.error, r.fit, r.old_fit, r.chol_info), tag
        else:
            for n, (Fg, Fr) in enumerate(zip(g.factors, r.factors)):
                assert rel_err(Fg, Fr) <= tol, tag + ": factor %d rel err %.3e" % (n, rel_err(Fg, Fr))
            assert rel_err(g.lam, r.lam) <= tol, tag + ": lambda rel err %.3e" % rel_err(g.lam, r.lam)
            assert abs(g.fit - r.fit) <= 1e-12, tag + ": fit %.17g != %.17g" % (g.fit, r.fit)


def _assert_vs_oracle(run, want, w, what):
    if w in LENIENT:
        same = [i for i, (g, r) in enumerate(zip(run.models, want.models)) if g.iters == r.iters]
        assert len(same) >= len(want.models) - 1, what
        assert_models_close([run.models[i] for i in same], [want.models[i] for i in same], want.x_norm, rtol=1e-7,
                            what=what)
    else:
        assert run.report["iter"] == want.iters, what
        assert_models_close(run.models, want.models, want.x_norm, what=what)
    assert run.report["n_ktensors"] == want.n_ktensors and run.report["ktensor_comp_sum"] == want.comp_sum, what
    assert abs(run.report["X_norm"] - want.x_norm) <= 1e-12 * want.x_norm, what


# ---------------------------------------------------------------------------------------------------------------------
# 1. knob and launch-path matrix
@pytest.mark.parametrize("w", MATRIX)
def test_default_path_vs_oracle(setting_results, oracle_results, w):
    _assert_vs_oracle(_result(setting_results, w, "default"), oracle_results(w), w, "%s default" % w)


def _default_period(w, workloads):
    X, ms, p = workloads[w]
    eligible = X.ndim == 3 and min(X.shape) >= 64 and not p.get("line_search") and p.get("mttkrp_method") != "mttkrp"
    return 2 if eligible else 1


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("w", MATRIX)
def test_path_matches_default(setting_results, oracle_results, workloads, w, path):
    if (w, _setting_of(path)) in SKIP:
        pytest.skip(SKIP[(w, _setting_of(path))])
    ref = _result(setting_results, w, "default")
    got = _result(setting_results, w, path)
    what = "%s %s" % (w, path)
    lenient = w in LENIENT and path in CLOSE
    # discrete outcomes
    assert ref.report["sweep_period"] == _default_period(w, workloads), what
    for f in ("n_ktensors", "ktensor_comp_sum"):
        assert got.report[f] == ref.report[f], "%s: %s %s != %s" % (what, f, got.report[f], ref.report[f])
    if not lenient:
        assert got.report["iter"] == ref.report["iter"], what
        assert np.array_equal(got.cols, ref.cols), what
        if (w, _setting_of(path)) in SCHEDULE_OFF:
            # the knob switched the multi-sweep schedule off: two contractions of 2 nX C flop per pass
            assert got.report["sweep_period"] == 1 and ref.report["sweep_period"] == 2, what
            nX = float(np.prod(workloads[w][0].shape))
            assert got.report["tensor_flops"] == 2.0 * nX * 2 * float(got.cols.astype(np.float64).sum()), what
        else:
            assert got.report["sweep_period"] == ref.report["sweep_period"], what
            assert got.report["tensor_flops"] == ref.report["tensor_flops"], what
    # results
    if lenient:
        same = [i for i, (g, r) in enumerate(zip(got.models, ref.models)) if g.iters == r.iters]
        assert len(same) >= len(ref.models) - 1, what
        assert_models_close([got.models[i] for i in same], [ref.models[i] for i in same],
                            oracle_results(w).x_norm, rtol=1e-7, what=what)
    else:
        _assert_close_or_equal(got, ref, path in BITWISE, 1e-11, what)
    if path in CLOSE:
        same = all(np.array_equal(F, G) for g, r in zip(got.models, ref.models) for F, G in zip(g.factors, r.factors))
        print("%s: bit-identical to the default path: %s" % (what, same))
        _assert_vs_oracle(got, oracle_results(w), w, what)


def _launch_delta(w, setting, workloads):
    """Change of kernel_launches against the default path for a forced, whole-queue, graphed run (exactly K + 1
    passes), from enqueue_iteration: the prefactor fork is one launch per mode; the fused reduction drops the reduce
    kernel of every mode with its own MTTKRP; the narrow tail adds its instance to every MTTKRP and pair contraction."""
    K = workloads[w][2]["max_iterations"]
    per_pass = {
        ("A", "prefactor"): 3, ("C", "prefactor"): 3, ("E", "prefactor"): 3,
        ("A", "pdl_prefactor"): 3, ("C", "pdl_prefactor"): 3, ("E", "pdl_prefactor"): 3,
        ("C", "fused_reduce"): -1, ("E", "fused_reduce"): -3,  # C: only mode 0 has its own MTTKRP
        ("C", "narrow"): 2, ("E", "narrow"): 3,  # C: mode 0's MTTKRP and the pair contraction of modes 1, 2
    }
    return per_pass.get((w, setting), 0) * (K + 1)


@pytest.mark.parametrize("setting", ["graph_batch_1", "graph_batch_4", "graph_batch_64", "pdl", "update_prof",
                                     "prefactor", "pdl_prefactor", "fused_reduce", "narrow"])
@pytest.mark.parametrize("w", ["A", "C", "E"])
def test_knob_changes_launches(setting_results, workloads, w, setting):
    """The knob took effect (or, for the launch mechanics, launched exactly what the default path launches)."""
    if (w, setting) in SCHEDULE_OFF:
        pytest.skip("the knob also switches the multi-sweep schedule off: the count follows another schedule")
    ref = _result(setting_results, w, "default").report["kernel_launches"]
    got = _result(setting_results, w, setting).report["kernel_launches"]
    assert got - ref == _launch_delta(w, setting, workloads), (w, setting, ref, got)


def test_update_prof_prints(setting_results):
    assert "[update prof] mode 0" in setting_results("update_prof")[1]
    assert "[update prof]" not in setting_results("default")[1]


def _kernels(setting_results, setting, w):
    names = setting_results(setting)[0]["%s|profile" % w].report["kernels"]
    assert names, "the profiler recorded nothing"
    return names


def _has(names, pattern):
    return any(re.search(pattern, n) for n in names)


def test_wm_max_kernels(setting_results):
    """WM_MAX=8 reaches mttkrp_dmma_kernel<8, 4, ...>, which the height rule never picks for these extents;
    WM_MAX=4 leaves only 4-row-group tiles."""
    default, k8, k4 = (_kernels(setting_results, s, "E") for s in ("default", "wm_max_8", "wm_max_4"))
    assert _has(default, r"mttkrp_dmma_kernel<6, 4, false>") and not _has(default, r"mttkrp_dmma_kernel<8, 4")
    assert _has(k8, r"mttkrp_dmma_kernel<8, 4, false>")
    assert _has(k4, r"mttkrp_dmma_kernel<4, 4, false>") and not _has(k4, r"mttkrp_dmma_kernel<[5-8], 4")


def test_narrow_kernels(setting_results):
    """NARROW launches the <..., true> column-tail instances; the default path never does."""
    for w in ("C", "E"):
        assert not _has(_kernels(setting_results, "default", w), r"mttkrp_dmma_kernel<\d, 4, true>"), w
        assert _has(_kernels(setting_results, "narrow", w), r"mttkrp_dmma_kernel<\d, 4, true>"), w
    assert not _has(_kernels(setting_results, "default", "C"), r"pair_gemm_kernel<\d, 4, true>")
    assert _has(_kernels(setting_results, "narrow", "C"), r"pair_gemm_kernel<\d, 4, true>")


def test_no_graph_launches(setting_results):
    """NO_GRAPH enqueues every kernel from the host; the default path replays graphs."""
    assert _has(_kernels(setting_results, "default", "E"), r"^cudaGraphLaunch")
    names = _kernels(setting_results, "no_graph", "E")
    assert not _has(names, r"^cudaGraphLaunch") and _has(names, r"^cudaLaunchKernel")


@pytest.mark.parametrize("path", ["default+timing", "no_graph+timing"])
@pytest.mark.parametrize("w", MATRIX)
def test_timing_report(setting_results, w, path):
    """The windows lie inside the run: both positive, their sum within the device time (event resolution ~1 us)."""
    r = _result(setting_results, w, path).report
    assert r["mttkrp_ms"] > 0 and r["update_ms"] > 0, r
    assert r["mttkrp_ms"] + r["update_ms"] <= r["device_ms"] * 1.001 + 0.01, r
    untimed = _result(setting_results, w, _setting_of(path)).report
    assert untimed["mttkrp_ms"] == 0 and untimed["update_ms"] == 0


def test_timing_wide_update_window(setting_results):
    """The wide kernels sit inside the update window: one rank-130 model's update takes far longer than one
    rank-20 model's (one B200, 1000 W power limit: 4.02 ms against 0.32 ms, a ratio of 12.6)."""
    res = setting_results("default")[0]
    wide, narrow = res["T130|timing"].report, res["T20|timing"].report
    ratio = wide["update_ms"] / narrow["update_ms"]
    print("update_ms rank 130 / rank 20: %.3f / %.3f = %.2f" % (wide["update_ms"], narrow["update_ms"], ratio))
    assert ratio > 4.0, (wide, narrow)


# ---------------------------------------------------------------------------------------------------------------------
# 2. state kept between calls in one Engine
def _fit(pkg, X, ms, params, engine=None, timing=0):
    kts = to_ktensors(pkg, ms)
    rep = pkg.cp_cals(X, kts, pkg.CalsParams(**params), engine=engine, timing=timing)
    return rep, kts


def _assert_identical(a, b, what):
    for i, (x, y) in enumerate(zip(a, b)):
        assert x.iters == y.iters, (what, i)
        for n, (Fx, Fy) in enumerate(zip(x.factors, y.factors)):
            assert np.array_equal(Fx, Fy), "%s model %d factor %d: rel %.3e" % (what, i, n, rel_err(Fx, Fy))
        assert np.array_equal(x.lam, y.lam), (what, i)
        assert (x.error, x.fit, x.old_fit, x.chol_info) == (y.error, y.fit, y.old_fit, y.chol_info), (what, i)


def _same_as_fresh(pkg, eng, X, ms, params, what, timing=0, check_norm=True):
    """Run in `eng` and on a fresh Engine: bit-identical results and reports; ||X|| from the current tensor."""
    import oracle
    rep, kts = _fit(pkg, X, ms, params, engine=eng, timing=timing)
    cols = eng.iteration_cols()
    rep0, kts0 = _fit(pkg, X, ms, params, timing=timing)
    _assert_identical(kts, kts0, what)
    for f in ("iter", "n_ktensors", "ktensor_comp_sum", "tensor_flops", "sweep_period", "X_norm"):
        assert getattr(rep, f) == getattr(rep0, f), (what, f)
    if check_norm:
        xn = oracle.norm(X)
        assert abs(rep.X_norm - xn) <= 1e-12 * xn, (what, rep.X_norm, xn)
    return rep, kts, cols


def _assert_rerun(eng, kts, rep, what):
    rep2 = eng.rerun()
    assert rep2.iter == rep.iter, what
    for (fs, lam, st), k in zip(eng.fetch_all(), kts):
        assert all(np.array_equal(F, G) for F, G in zip(fs, k.factors)), what
        assert np.array_equal(lam, k.lam) and st.iters == k.iters and st.error == k.error, what


def test_engine_state_tensor_changes(pkg):
    """New contents at the same shape (the (2, 0, 1) copy Xr, the odd-extent staging block, the 4-mode Xq, the cached
    ||X||, the kept plans and graphs), another shape, and back."""
    rng = np.random.default_rng(201)
    p3 = dict(max_iterations=4, buffer_size=20, force_max_iter=True)
    shapes = [(72, 66, 64), (72, 66, 64), (67, 64, 65), (67, 64, 65), (20, 44, 9, 31), (20, 44, 9, 31), (72, 66, 64)]
    Xs = [rng.uniform(-1, 1, size=s) for s in shapes]
    Xs[-1] = Xs[0]
    models = {}
    with pkg.Engine(0) as eng:
        for k, (s, X) in enumerate(zip(shapes, Xs)):
            if s not in models:
                models[s] = caseio.random_models(rng, s, [3, 7, 1, 5, 4, 6])
            rep, kts, _ = _same_as_fresh(pkg, eng, X, models[s], p3, "tensor %d %s" % (k, s))
            if len(s) == 3:
                assert rep.sweep_period == 2
            if k in (1, 3, 5):
                _assert_rerun(eng, kts, rep, "rerun after tensor %d" % k)


def test_engines_share_kernel_limits(pkg):
    """A second Engine with a smaller problem between two calls of the first: the shared-memory limits of the kernels
    belong to the process, so the second one must not lower a limit the first one still launches with."""
    rng = np.random.default_rng(205)
    big, small = (72, 66, 64), (20, 44, 9, 31)
    Xb, Xs = rng.uniform(-1, 1, size=big), rng.uniform(-1, 1, size=small)
    mb, msm = caseio.random_models(rng, big, [12, 9]), caseio.random_models(rng, small, [3, 2])
    p = dict(max_iterations=3, buffer_size=21, force_max_iter=True)
    with pkg.Engine(0) as eng:
        first = _fit(pkg, Xb, mb, p, engine=eng)[1]
        _fit(pkg, Xs, msm, p)
        _assert_identical(_fit(pkg, Xb, mb, p, engine=eng)[1], first, "after a smaller problem on another Engine")


def test_engine_state_settings_alternate(pkg, monkeypatch):
    """Settings that change from call to call in one Engine: timing, the MTTKRP schedule, the per-call knobs MSDT and
    FUSED_LEAF, NNLS (with carried active sets) then unconstrained, line search on then off."""
    rng = np.random.default_rng(202)
    modes = (72, 66, 64)
    gen = [rng.uniform(0, 1, size=(i, 3)) for i in modes]
    X = caseio.ktensor_to_tensor(gen, np.ones(3)) + 0.05 * rng.uniform(0, 1, size=modes)
    ms = caseio.random_models(rng, modes, [3, 7, 1, 12, 5, 9, 2])
    base = dict(max_iterations=4, force_max_iter=True)
    steps = [
        ("timing", {}, dict(buffer_size=39), 1),
        ("untimed", {}, dict(buffer_size=39), 0),
        ("queueing timed", {}, dict(buffer_size=14), 1),
        ("per-mode", {}, dict(buffer_size=39, mttkrp_method="mttkrp"), 0),
        ("auto", {}, dict(buffer_size=39), 0),
        ("msdt 0", {"CALS_B200_MSDT": "0"}, dict(buffer_size=39), 0),
        ("msdt 1", {"CALS_B200_MSDT": "1"}, dict(buffer_size=39), 0),
        ("fused leaf 0", {"CALS_B200_FUSED_LEAF": "0"}, dict(buffer_size=39), 0),
        ("fused leaf 1", {"CALS_B200_FUSED_LEAF": "1"}, dict(buffer_size=39), 0),
        ("nnls", {}, dict(buffer_size=14, update_method="nnls"), 0),
        ("unconstrained", {}, dict(buffer_size=14), 0),
        ("line search", {}, dict(buffer_size=14, line_search=True, line_search_interval=3), 0),
        ("no line search", {}, dict(buffer_size=14), 0),
    ]
    with pkg.Engine(0) as eng:
        for what, env, extra, timing in steps:
            for k in ("CALS_B200_MSDT", "CALS_B200_FUSED_LEAF"):
                monkeypatch.delenv(k, raising=False)
            for k, v in env.items():
                monkeypatch.setenv(k, v)
            params = dict(base, **extra)
            rep, kts, _ = _same_as_fresh(pkg, eng, X, ms, params, what, timing=timing)
            if what in ("untimed", "msdt 1", "no line search"):
                _assert_rerun(eng, kts, rep, "rerun after " + what)
            if what == "nnls":  # a second NNLS call that starts from the active sets the first one left
                kts_e = to_ktensors(pkg, ms)
                kts_f = to_ktensors(pkg, ms)
                for a, b, k in zip(kts_e, kts_f, kts):
                    a.active_set = [s.copy() for s in k.active_set]
                    b.active_set = [s.copy() for s in k.active_set]
                pkg.cp_cals(X, kts_e, pkg.CalsParams(**params), engine=eng)
                pkg.cp_cals(X, kts_f, pkg.CalsParams(**params))
                _assert_identical(kts_e, kts_f, "nnls with carried active sets")


def test_engine_state_rank_sequence(pkg):
    """A queue with wide models, one without (the narrow kernel and the prefactor scratch sized again), and back."""
    rng = np.random.default_rng(203)
    modes = (66, 64, 70)
    X = rng.uniform(-1, 1, size=modes)
    seqs = [[130, 7, 20], [7, 20, 3], [130, 7, 20], [97, 5], [7, 20, 3]]
    models = {}
    with pkg.Engine(0) as eng:
        for k, ranks in enumerate(seqs):
            key = tuple(ranks)
            if key not in models:
                models[key] = caseio.random_models(rng, modes, ranks)
            rep, kts, _ = _same_as_fresh(pkg, eng, X, models[key], dict(max_iterations=3, buffer_size=sum(ranks),
                                                                        force_max_iter=True), "ranks %s" % ranks)
            if k == 2:
                _assert_rerun(eng, kts, rep, "rerun, ranks %s" % ranks)


def test_set_tensor_dev_matches_host_upload(pkg):
    """set_tensor_dev from a torch CUDA tensor gives the same run as set_tensor of the same values."""
    import torch
    rng = np.random.default_rng(204)
    modes = (67, 64, 65)
    X = rng.uniform(-1, 1, size=modes)
    ms = caseio.random_models(rng, modes, [3, 7, 1, 5])
    p = pkg.CalsParams(max_iterations=4, buffer_size=16, force_max_iter=True)
    ref = to_ktensors(pkg, ms)
    pkg.cp_cals(X, ref, p)
    Xd = torch.from_numpy(np.asfortranarray(X).ravel(order="F").copy()).to("cuda:0")
    torch.cuda.synchronize()
    with pkg.Engine(0) as eng:
        eng.set_tensor_dev(Xd.data_ptr(), modes)
        kts = to_ktensors(pkg, ms)  # cp_cals would upload X from the host: drive the engine directly
        eng.configure(p.buffer_size, p.max_iterations, p.tol, force_max_iter=True)
        eng.set_line_search(False)
        eng.set_timing(0)
        eng.set_pair_node(True)
        eng.clear_models()
        eng.enqueue_many([k.factors for k in kts])
        rep = eng.run()
        out = eng.fetch_all()
        assert rep.iter == 4
    for (fs, lam, st), k in zip(out, ref):
        assert all(np.array_equal(F, G) for F, G in zip(fs, k.factors))
        assert np.array_equal(lam, k.lam) and st.error == k.error and st.fit == k.fit
    del Xd


# ---------------------------------------------------------------------------------------------------------------------
# 3. two GPUs: a sharded model set with a wide model
def _sharded_case():
    rng = np.random.default_rng(301)
    modes = (40, 36, 34)
    X = rng.uniform(-1, 1, size=modes)
    return X, caseio.random_models(rng, modes, [130, 7, 20, 3, 12])


def _sharded_worker(rank, world, port, out_dir):
    for p in (os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
        sys.path.insert(0, p)
    import torch
    import torch.distributed as dist
    from conftest import load_package
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        pkg = load_package()
        import importlib
        d = importlib.import_module("cp_cals_b200.distributed")
        X, ms = _sharded_case()
        kts = to_ktensors(pkg, ms)
        d.cp_cals_sharded(X, kts, pkg.CalsParams(max_iterations=4, buffer_size=150, force_max_iter=True), device=rank,
                          gather_device=torch.device("cuda", rank))
        np.savez(os.path.join(out_dir, "wide_rank%d.npz" % rank),
                 **{"m%d_f%d" % (i, n): F for i, k in enumerate(kts) for n, F in enumerate(k.factors)},
                 **{"m%d_lam" % i: k.lam for i, k in enumerate(kts)},
                 **{"m%d_st" % i: np.array([k.iters, k.error, k.fit]) for i, k in enumerate(kts)})
    finally:
        dist.destroy_process_group()


def test_two_gpus_sharded_wide_model(pkg, tmp_path):
    import socket

    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_sharded_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    X, ms = _sharded_case()
    one = to_ktensors(pkg, ms)
    pkg.cp_cals(X, one, pkg.CalsParams(max_iterations=4, buffer_size=150, force_max_iter=True), device=0)
    outs = [np.load(os.path.join(str(tmp_path), "wide_rank%d.npz" % r)) for r in range(2)]
    for k in outs[0].files:  # every rank holds every fitted model
        assert np.array_equal(outs[0][k], outs[1][k]), k
    for i, k in enumerate(one):
        for n in range(X.ndim):
            assert rel_err(outs[0]["m%d_f%d" % (i, n)], k.factors[n]) <= 1e-11, (i, n)
        assert rel_err(outs[0]["m%d_lam" % i], k.lam) <= 1e-11, i
        st = outs[0]["m%d_st" % i]
        assert int(st[0]) == k.iters and abs(st[2] - k.fit) <= 1e-12, i


if __name__ == "__main__":
    if len(sys.argv) != 4 or sys.argv[1] != "--worker":
        sys.exit("usage: python tests/test_launch_paths.py --worker CASES.npz OUT.npz")
    _worker(sys.argv[2], sys.argv[3])
