"""Shared helpers for the parity tests (test infrastructure)."""
import os

import numpy as np

import caseio

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# north_star tolerance: per-iteration fit and factor matrices within 1e-9 relative error in FP64
RTOL = 1e-9


def load_golden(name):
    """Returns (X, models_in, models_ref, params, report) from tests/golden/<name>.npz."""
    d = np.load(os.path.join(GOLDEN, name + ".npz"))
    X = d["X"]
    N = X.ndim
    ins, refs = [], []
    for i in range(int(d["n_models"])):
        jk = d["m%d_jk" % i]
        st = d["m%d_stats" % i]
        ins.append(caseio.Model(factors=[np.asfortranarray(d["m%d_in%d" % (i, n)]) for n in range(N)],
                                jk_mode=int(jk[0]), jk_fiber=int(jk[1])))
        refs.append(caseio.Model(factors=[d["m%d_out%d" % (i, n)] for n in range(N)], lam=d["m%d_lam" % i],
                                 jk_mode=int(jk[0]), jk_fiber=int(jk[1]), iters=int(st[0]), error=float(st[1]),
                                 fit_diff=float(st[2])))
    params = {k[len("param_"):]: d[k].item() for k in d.files if k.startswith("param_")}
    report = {k: d[k].item() for k in ("iter", "n_ktensors", "comp_sum", "x_norm")}
    return X, ins, refs, params, report


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    den = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / den) if den > 0 else float(np.linalg.norm(a - b))


def assert_models_close(got, ref, x_norm, rtol=RTOL, check_iters=True, what=""):
    """got/ref: sequences of objects with .factors .lam .iters .error.  The error is a cancellation
    (||X||^2 + t2 - 2 t3), so it is compared relative to ||X|| (i.e. through the fit), never relative to itself
    (SURVEY.md section 8c)."""
    assert len(got) == len(ref)
    for i, (g, r) in enumerate(zip(got, ref)):
        tag = "%s model %d (rank %d)" % (what, i, r.factors[0].shape[1])
        if check_iters:
            assert int(g.iters) == int(r.iters), tag + ": iters %d != %d" % (g.iters, r.iters)
        for n, (Fg, Fr) in enumerate(zip(g.factors, r.factors)):
            e = rel_err(Fg, Fr)
            assert e <= rtol, tag + ": factor %d rel err %.3e" % (n, e)
        e = rel_err(g.lam, r.lam)
        assert e <= rtol, tag + ": lambda rel err %.3e" % e
        e = abs(g.error - r.error) / x_norm
        assert e <= rtol, tag + ": |d error|/||X|| = %.3e" % e


def load_sampled(name):
    """tests/golden/<name>.npz written by oracle/make_golden.py's pack_sampled."""
    d = np.load(os.path.join(GOLDEN, name + ".npz"))
    return {k: (d[k].item() if d[k].ndim == 0 else d[k]) for k in d.files}


def assert_sampled_models_close(got, want, rtol=RTOL, what=""):
    """got: objects with .factors .lam .iters .error .fit in queue order; want: load_sampled().  Per model, the stored
    column's sampled rows of every factor within rtol of that whole column's norm, its lambda entry within rtol, the
    error within rtol of ||X|| (a cancellation, see assert_models_close), the fit within rtol, equal iteration counts."""
    cols = want["cols"]
    assert len(got) == len(cols)
    xn = want["x_norm"]
    for i, (g, c) in enumerate(zip(got, cols)):
        tag = "%s model %d (rank %d)" % (what, i, g.factors[0].shape[1])
        assert int(g.iters) == int(want["iters"][i]), tag + ": iters %d != %d" % (g.iters, want["iters"][i])
        for n, F in enumerate(g.factors):
            e = np.abs(F[want["rows%d" % n], c] - want["f%d" % n][i]).max() / want["colnorm%d" % n][i]
            assert e <= rtol, tag + ": factor %d column %d sampled rel err %.3e" % (n, c, e)
        e = abs(g.lam[c] - want["lam"][i]) / abs(want["lam"][i])
        assert e <= rtol, tag + ": lambda rel err %.3e" % e
        assert abs(g.error - want["error"][i]) / xn <= rtol, tag + ": |d error|/||X|| = %.3e" % (
            abs(g.error - want["error"][i]) / xn)
        assert abs(g.fit - want["fit"][i]) <= rtol, tag + ": fit %.15f != %.15f" % (g.fit, want["fit"][i])


def to_ktensors(pkg, models):
    return [pkg.Ktensor([np.array(F, order="F", copy=True) for F in m.factors], None, m.jk_mode, m.jk_fiber)
            for m in models]
