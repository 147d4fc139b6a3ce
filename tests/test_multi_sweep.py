"""Multi-sweep dimension tree (3 modes, csrc/engine.cu: run_loop; csrc/pairnode.cuh).

Even iterations contract modes 2 and 1, odd iterations mode 0; the mode-1 contraction of an even iteration also serves
mode 0 of the next one, unless the scheduler moves columns in between (then mode 0 runs its own MTTKRP).  Every mode
sees the factors of the per-mode MTTKRP, so the results equal the one-sweep schedule's up to the association of the
sums.  CALS_B200_MSDT=0/1 forces either schedule.
"""
import math

import numpy as np
import pytest

import caseio
import oracle
from helpers import assert_models_close, rel_err, to_ktensors

pytestmark = pytest.mark.gpu


def run(pkg, monkeypatch, msdt, X, ms, engine=None, **params):
    if msdt is None:
        monkeypatch.delenv("CALS_B200_MSDT", raising=False)
    else:
        monkeypatch.setenv("CALS_B200_MSDT", msdt)
    kts = to_ktensors(pkg, ms)
    rep = pkg.cp_cals(X, kts, pkg.CalsParams(**params), engine=engine)
    return rep, kts


def assert_schedules_equal(a, b, tol=1e-11, what=""):
    for i, (ka, kb) in enumerate(zip(a, b)):
        assert ka.iters == kb.iters, (what, i)
        for n, (Fa, Fb) in enumerate(zip(ka.factors, kb.factors)):
            assert rel_err(Fa, Fb) <= tol, "%s model %d factor %d: %.3e" % (what, i, n, rel_err(Fa, Fb))
        assert rel_err(ka.lam, kb.lam) <= tol, (what, i)
        assert abs(ka.fit - kb.fit) <= 1e-12, (what, i)


@pytest.mark.parametrize("modes,ranks", [
    ((37, 45, 23), [4, 9, 1, 12, 7]),      # K tail on every contracted mode (KT = 40), no extent a multiple of 8
    ((83, 41, 50), [3, 5, 2]),             # several K tiles, i-extents off the tile heights
    ((40, 56, 24), [20] * 13 + [3]),       # 263 columns: ragged last octet, two n-tiles
    ((24, 20, 12), [16] * 20 + [7]),       # 327 columns: two n-tiles of 3 octets, 7 columns in the last
])
def test_multi_sweep_parity(pkg, monkeypatch, modes, ranks):
    """Forced K = 1 .. 6, so that runs end on both parities: against the one-sweep schedule (1e-11) and the oracle."""
    rng = np.random.default_rng(hash((modes, 31)) % 2 ** 32)
    X = rng.uniform(-1, 1, size=modes)
    ms = caseio.random_models(rng, modes, ranks)
    bs = sum(ranks)
    with pkg.Engine(0) as eng:
        for K in range(1, 7):
            want = oracle.cp_cals(X, ms, max_iter=K, force_max_iter=True, buffer_size=bs)
            out = {}
            for msdt in ("0", "1"):
                rep, kts = run(pkg, monkeypatch, msdt, X, ms, engine=eng, max_iterations=K, buffer_size=bs,
                               force_max_iter=True)
                assert rep.pair_node and rep.sweep_period == (2 if msdt == "1" else 1)
                assert rep.iter == want.iters
                assert_models_close(kts, want.models, want.x_norm, what="msdt=%s K=%d" % (msdt, K))
                out[msdt] = kts
            assert_schedules_equal(out["1"], out["0"], what="K=%d" % K)


@pytest.mark.parametrize("modes,ranks", [
    ((37, 45, 23), [4, 9, 1, 12, 7]),      # first leaves as their own pass over T, TMA-fed (narrow grid)
    ((24, 20, 12), [20] * 30 + [3]),       # 603 columns: the plain slow-leaf kernel
])
def test_multi_sweep_separate_first_leaf(pkg, monkeypatch, modes, ranks):
    """CALS_B200_FUSED_LEAF=0 (the default of narrow buffers over a large T, e.g. the 8-way shard of config 2): every
    node's first leaf streams T in a pass of its own."""
    monkeypatch.setenv("CALS_B200_FUSED_LEAF", "0")
    rng = np.random.default_rng(hash((modes, 32)) % 2 ** 32)
    X = rng.uniform(-1, 1, size=modes)
    ms = caseio.random_models(rng, modes, ranks)
    bs = sum(ranks)
    for K in (3, 4):
        want = oracle.cp_cals(X, ms, max_iter=K, force_max_iter=True, buffer_size=bs)
        rep, kts = run(pkg, monkeypatch, "1", X, ms, max_iterations=K, buffer_size=bs, force_max_iter=True)
        assert rep.sweep_period == 2 and rep.iter == want.iters
        assert_models_close(kts, want.models, want.x_norm, what="separate leaf K=%d" % K)


def test_flop_counter_whole_queue(pkg, monkeypatch):
    """Whole queue resident, forced K: K + ceil(K/2) contractions of 2 * nX * C flop."""
    rng = np.random.default_rng(5)
    modes = (30, 26, 22)
    ranks = [3, 7, 5]
    X = rng.uniform(-1, 1, size=modes)
    ms = caseio.random_models(rng, modes, ranks)
    nX, C = float(np.prod(modes)), sum(ranks)
    for K in range(1, 6):
        rep, _ = run(pkg, monkeypatch, "1", X, ms, max_iterations=K, buffer_size=C, force_max_iter=True)
        assert rep.tensor_flops == 2.0 * nX * C * (K + math.ceil(K / 2)), K
        rep, _ = run(pkg, monkeypatch, "0", X, ms, max_iterations=K, buffer_size=C, force_max_iter=True)
        assert rep.tensor_flops == 2.0 * nX * C * 2 * K, K


def forced_queue_passes(ranks, K, buffer):
    """(columns, columns moved) of every pass of a forced-K run with FIFO admission (csrc/sched.cuh): a model admitted
    in pass a is updated in passes a .. a+K-1 and evicted by the scheduler of pass a+K."""
    live, nxt, p, out = [], 0, 0, []
    while True:
        keep = [(m, a) for m, a in live if p - a < K]
        changed = len(keep) != len(live)
        live = keep
        col = sum(ranks[m] for m, _ in live)
        while nxt < len(ranks) and col + ranks[nxt] <= buffer:
            live.append((nxt, p))
            col += ranks[nxt]
            nxt += 1
            changed = True
        if not live:
            return out
        out.append((col, changed))
        p += 1


def test_queue_changes_fall_back(pkg, monkeypatch):
    """A buffer smaller than the queue: models are evicted and admitted on odd passes too.  There the carried T does not
    match the columns and mode 0 runs its own MTTKRP -- one more contraction for every such pass."""
    rng = np.random.default_rng(21)
    modes = (40, 41, 29)
    ranks = [3, 8, 2, 5, 4, 6, 1, 7]
    K, bs = 5, 12
    X = rng.uniform(-1, 1, size=modes)
    ms = caseio.random_models(rng, modes, ranks)
    want = oracle.cp_cals(X, ms, max_iter=K, force_max_iter=True, buffer_size=bs)
    with pkg.Engine(0) as eng:
        rep, kts = run(pkg, monkeypatch, "1", X, ms, engine=eng, max_iterations=K, buffer_size=bs, force_max_iter=True)
        cols = eng.iteration_cols()
    assert rep.sweep_period == 2 and rep.iter == want.iters
    assert_models_close(kts, want.models, want.x_norm, what="queue")
    passes = forced_queue_passes(ranks, K, bs)
    assert [c for c, _ in passes] == list(cols)
    assert any(ch for p, (_, ch) in enumerate(passes) if p % 2 == 1)  # the fallback did run
    expect = sum(c * (2 if p % 2 == 0 else 1 + int(ch)) for p, (c, ch) in enumerate(passes))
    assert rep.tensor_flops == 2.0 * float(np.prod(modes)) * expect


def test_always_evict_first(pkg, monkeypatch):
    """ALWAYS_EVICT_FIRST moves columns in every pass: every odd pass falls back to the full MTTKRP of mode 0."""
    rng = np.random.default_rng(22)
    modes = (23, 30, 17)
    ranks = [2, 4, 3, 5, 1]
    X = rng.uniform(-1, 1, size=modes)
    ms = caseio.random_models(rng, modes, ranks)
    want = oracle.cp_cals(X, ms, max_iter=6, force_max_iter=True, buffer_size=9, always_evict_first=True)
    with pkg.Engine(0) as eng:
        rep, kts = run(pkg, monkeypatch, "1", X, ms, engine=eng, max_iterations=6, buffer_size=9, force_max_iter=True,
                       always_evict_first=True)
        cols = eng.iteration_cols().astype(np.float64)
    assert rep.sweep_period == 2 and rep.iter == want.iters
    assert_models_close(kts, want.models, want.x_norm, what="evict first")
    assert rep.tensor_flops == 2.0 * float(np.prod(modes)) * 2 * cols.sum()


def test_tol_eviction(pkg, monkeypatch):
    """tol-based stopping with queueing: models leave whenever they converge, on either parity."""
    rng = np.random.default_rng(23)
    modes = (30, 28, 26)
    gen = [rng.uniform(0, 1, size=(i, 3)) for i in modes]
    X = caseio.ktensor_to_tensor(gen, np.ones(3)) + 0.01 * rng.standard_normal(modes)
    ranks = [1, 2, 3, 4, 2, 3, 1, 5]
    ms = caseio.random_models(rng, modes, ranks)
    want = oracle.cp_cals(X, ms, max_iter=60, tol=1e-5, buffer_size=9)
    rep, kts = run(pkg, monkeypatch, "1", X, ms, max_iterations=60, tol=1e-5, buffer_size=9)
    assert rep.sweep_period == 2
    same = [i for i, (g, r) in enumerate(zip(kts, want.models)) if g.iters == r.iters]
    assert len(same) >= len(ranks) - 1
    assert_models_close([kts[i] for i in same], [want.models[i] for i in same], want.x_norm, rtol=1e-7, what="tol")


def test_jackknife_and_nnls(pkg, monkeypatch):
    """Flagged (jackknife) models and the NNLS update give the same results under both schedules."""
    rng = np.random.default_rng(24)
    modes = (21, 19, 16)
    gen = [rng.uniform(0, 1, size=(i, 3)) for i in modes]
    X = caseio.ktensor_to_tensor(gen, np.ones(3)) + 0.05 * rng.standard_normal(modes)
    ms = caseio.random_models(rng, modes, [2, 3, 4, 3])
    ms[1].jk_mode, ms[1].jk_fiber = 0, 5
    ms[3].jk_mode, ms[3].jk_fiber = 0, 20
    for extra in (dict(), dict(update_method="nnls")):
        out = {}
        for msdt in ("0", "1"):
            rep, out[msdt] = run(pkg, monkeypatch, msdt, X, ms, max_iterations=7, buffer_size=12, force_max_iter=True,
                                 **extra)
            assert rep.sweep_period == (2 if msdt == "1" else 1)
        assert_schedules_equal(out["1"], out["0"], tol=1e-9, what=str(extra))


def test_gate(pkg, monkeypatch):
    """By default the schedule runs on 3-mode tensors whose extents are all at least 64; never with line search or on
    4 modes, even when forced."""
    rng = np.random.default_rng(25)

    def period(modes, msdt=None, **extra):
        X = rng.uniform(-1, 1, size=modes)
        ms = caseio.random_models(rng, modes, [2, 3])
        rep, _ = run(pkg, monkeypatch, msdt, X, ms, max_iterations=4, buffer_size=5, force_max_iter=True, **extra)
        assert rep.pair_node
        return rep.sweep_period

    assert period((70, 66, 64)) == 2
    assert period((70, 66, 41)) == 1
    assert period((70, 66, 41), "1") == 2
    assert period((70, 66, 64), "0") == 1
    assert period((70, 66, 64), "1", line_search=True, line_search_interval=3) == 1
    assert period((12, 9, 8, 7), "1") == 1


def test_deterministic(pkg, monkeypatch):
    rng = np.random.default_rng(26)
    modes = (37, 45, 23)
    X = rng.uniform(-1, 1, size=modes)
    ms = caseio.random_models(rng, modes, [4, 9, 1, 12, 7])
    runs = [run(pkg, monkeypatch, "1", X, ms, max_iterations=5, buffer_size=33, force_max_iter=True)[1]
            for _ in range(2)]
    for a, b in zip(*runs):
        for Fa, Fb in zip(a.factors, b.factors):
            assert np.array_equal(Fa, Fb)
        assert np.array_equal(a.lam, b.lam)
