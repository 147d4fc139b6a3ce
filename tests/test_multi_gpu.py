"""N > 1 host logic (SURVEY 8e) on the CPU: world_size-2 gloo process groups exercise cp-cals_b200/distributed.py
(sharding plan, packing, the all-gather of results, jackknife sub-model sharding) with the oracle standing in for the
per-rank CUDA loop.  The -m gpu variant runs the real engine on as many GPUs as the box has."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _oracle_fit(X, kts, params, **kw):
    """Stand-in for cp_cals on one rank: the CPU oracle (test infrastructure) writing results back into the Ktensors."""
    import caseio
    import oracle
    ms = [caseio.Model(factors=[F.copy() for F in k.factors], jk_mode=k.jk_mode, jk_fiber=k.jk_fiber) for k in kts]
    res = oracle.cp_cals(X, ms, max_iter=params.max_iterations, tol=params.tol, buffer_size=params.buffer_size,
                         force_max_iter=params.force_max_iter)
    for k, r in zip(kts, res.models):
        k.factors, k.lam, k.iters, k.error, k.fit, k.old_fit = r.factors, r.lam, r.iters, r.error, r.fit, r.old_fit
    return res


def _case():
    rng = np.random.default_rng(42)
    modes = (9, 8, 7)
    X = rng.uniform(-1, 1, size=modes)
    ranks = [3, 1, 4, 1, 5, 2, 6, 2]
    import caseio
    return X, modes, ranks, caseio.random_models(rng, modes, ranks)


def _worker(rank, world, port, backend, use_engine, out_dir):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch
    import torch.distributed as dist
    from conftest import load_package
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    device = None
    if backend == "nccl":
        torch.cuda.set_device(rank)
        device = torch.device("cuda", rank)
    dist.init_process_group(backend, rank=rank, world_size=world)
    try:
        pkg = load_package()
        import importlib
        d = importlib.import_module("cp_cals_b200.distributed")
        X, modes, ranks, ms = _case()
        kts = [pkg.Ktensor([F.copy() for F in m.factors]) for m in ms]
        params = pkg.CalsParams(max_iterations=6, buffer_size=9, force_max_iter=True)
        kw = dict(device=rank, gather_device=device) if use_engine else dict(fit_fn=_oracle_fit)
        rep, mine = d.cp_cals_sharded(X, kts, params, **kw)
        np.savez(os.path.join(out_dir, "cals_rank%d.npz" % rank), mine=np.array(mine),
                 **{"m%d_f%d" % (i, n): F for i, k in enumerate(kts) for n, F in enumerate(k.factors)},
                 **{"m%d_lam" % i: k.lam for i, k in enumerate(kts)},
                 **{"m%d_st" % i: np.array([k.iters, k.error, k.fit]) for i, k in enumerate(kts)})
        # jackknife: the leave-one-out sub-models are what is sharded
        bases = [pkg.Ktensor([F.copy() for F in m.factors], m.lam.copy()) for m in ms[:2]]
        rep, groups = d.jk_cp_cals_sharded(X, bases, params, **kw)
        np.savez(os.path.join(out_dir, "jk_rank%d.npz" % rank),
                 **{"b%d_i%d_f%d" % (b, i, n): F for b, g in enumerate(groups) for i, k in enumerate(g)
                    for n, F in enumerate(k.factors)})
        dist.barrier()
    finally:
        dist.destroy_process_group()


def _spawn(world, backend, use_engine, tmp_path):
    import torch.multiprocessing as mp
    port = _free_port()
    mp.spawn(_worker, args=(world, port, backend, use_engine, str(tmp_path)), nprocs=world, join=True)


def _check_outputs(tmp_path, world, rtol):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import caseio
    import oracle
    X, modes, ranks, ms = _case()
    outs = [np.load(os.path.join(tmp_path, "cals_rank%d.npz" % r)) for r in range(world)]
    # the shards partition the model set
    all_mine = sorted(int(i) for o in outs for i in o["mine"])
    assert all_mine == list(range(len(ranks)))
    # every rank holds every fitted model, identical across ranks, and equal to fitting each shard alone
    from conftest import load_package
    d = __import__("importlib").import_module("cp_cals_b200.distributed") if load_package() else None
    parts = d.shard_models(ranks, world)
    for r, p in enumerate(parts):
        assert sorted(int(i) for i in outs[r]["mine"]) == p
        want = oracle.cp_cals(X, [ms[i] for i in p], max_iter=6, buffer_size=9, force_max_iter=True)
        for i, w in zip(p, want.models):
            for o in outs:
                for n in range(len(modes)):
                    a = o["m%d_f%d" % (i, n)]
                    assert np.linalg.norm(a - w.factors[n]) <= rtol * np.linalg.norm(w.factors[n])
                assert np.linalg.norm(o["m%d_lam" % i] - w.lam) <= rtol * np.linalg.norm(w.lam)
                st = o["m%d_st" % i]
                assert int(st[0]) == w.iters and abs(st[2] - w.fit) <= rtol
    jk = [np.load(os.path.join(tmp_path, "jk_rank%d.npz" % r)) for r in range(world)]
    for k in jk[0].files:
        for o in jk[1:]:
            assert np.array_equal(jk[0][k], o[k], equal_nan=True)
    assert len(jk[0].files) == 2 * modes[0] * len(modes)


def test_shard_models_plan(pkg):
    import importlib
    d = importlib.import_module("cp_cals_b200.distributed")
    ranks = [r for r in range(1, 21) for _ in range(10)]
    for world in (1, 2, 4, 8):
        parts = d.shard_models(ranks, world)
        assert sorted(i for p in parts for i in p) == list(range(len(ranks)))
        assert all(p == sorted(p) for p in parts)  # FIFO order inside a shard
        loads = [sum(ranks[i] for i in p) for p in parts]
        assert max(loads) - min(loads) <= 2  # largest rank first: BASELINE config 2 splits to within two columns
    for cfg_ranks in ([r for r in range(1, 31) for _ in range(5)], [r for r in (3, 5, 7, 9) for _ in range(299)]):
        loads = [sum(cfg_ranks[i] for i in p) for p in d.shard_models(cfg_ranks, 8)]  # configs 4 and 3
        assert max(loads) - min(loads) <= 3, loads
    assert d.shard_slabs(1000, 8) == [(0, 126), (126, 250), (250, 376), (376, 500), (500, 626), (626, 750), (750, 876),
                                      (876, 1000)]
    assert d.shard_slabs(7, 3) == [(0, 2), (2, 4), (4, 7)]
    assert all(lo % 2 == 0 for lo, _ in d.shard_slabs(299, 8))


def test_pack_unpack_roundtrip(pkg):
    import importlib
    d = importlib.import_module("cp_cals_b200.distributed")
    rng = np.random.default_rng(0)
    ms = [pkg.Ktensor([np.asfortranarray(rng.uniform(-1, 1, size=(i, r))) for i in (5, 4, 3)], rng.uniform(size=r))
          for r in (2, 1, 3)]
    for i, m in enumerate(ms):
        m.iters, m.error, m.fit, m.old_fit, m.chol_info = 3 + i, 0.5 * i, 0.9, 0.8, i
    buf = d.pack_models(ms)
    assert buf.size == d.packed_size(ms)
    blank = [pkg.Ktensor([np.zeros_like(F) for F in m.factors]) for m in ms]
    d.unpack_models(buf, blank)
    for a, b in zip(ms, blank):
        assert all(np.array_equal(x, y) for x, y in zip(a.factors, b.factors)) and np.array_equal(a.lam, b.lam)
        assert (a.iters, a.error, a.fit, a.old_fit, a.chol_info) == (b.iters, b.error, b.fit, b.old_fit, b.chol_info)


def test_world2_gloo_sharded_cp_cals_and_jackknife(tmp_path):
    _spawn(2, "gloo", False, tmp_path)
    _check_outputs(str(tmp_path), 2, 1e-12)


@pytest.mark.gpu
def test_multi_gpu_nccl_sharded_cp_cals(tmp_path):
    import torch
    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    _spawn(world, "nccl", True, tmp_path)
    _check_outputs(str(tmp_path), world, 1e-9)


# ---------------------------------------------------------------------------------------------------------------------
# Tensor sliced along one mode (BASELINE config 5)
@pytest.mark.gpu
@pytest.mark.parametrize("modes,C", [((14, 12, 10), 21), ((9, 8, 6, 10), 70), ((40, 18, 26), 300)])
@pytest.mark.parametrize("variant", ["naive", "dmma"])
def test_slab_partial_mttkrps_add_up(pkg, modes, C, variant):
    """One GPU, ranks emulated one after the other: for every sliced mode s and every output mode n, the partial
    MTTKRPs of the slabs add up to the MTTKRP of the whole tensor (n != s), or tile its rows (n == s)."""
    import importlib
    import oracle
    d = importlib.import_module("cp_cals_b200.distributed")
    rng = np.random.default_rng(sum(modes) + C)
    X = rng.uniform(-1, 1, size=modes)
    fs = [np.asfortranarray(rng.uniform(-1, 1, size=(i, C))) for i in modes]
    want = [oracle.mttkrp(X, fs, n) for n in range(len(modes))]
    v = pkg.MTTKRP_NAIVE if variant == "naive" else pkg.MTTKRP_DMMA
    W = 3
    for s in range(len(modes)):
        cuts = [0] + [hi for _, hi in d.shard_slabs(modes[s], W)]
        acc = [np.zeros_like(w) for w in want]
        for r in range(W):
            with pkg.Engine(0) as eng:
                eng.comm_alloc(r, W, d.exchange_capacity(modes, C))
                sl = [slice(None)] * len(modes)
                sl[s] = slice(cuts[r], cuts[r + 1])
                eng.set_tensor_slab(modes, s, cuts, X[tuple(sl)])
                assert abs(eng.tensor_norm() - np.linalg.norm(X[tuple(sl)])) <= 1e-12 * np.linalg.norm(X)
                for n in range(len(modes)):
                    part, _ = eng.mttkrp(fs, n, variant=v)
                    if n == s:  # only this slab's rows are produced, the rest stays zero
                        outside = np.ones(modes[n], dtype=bool)
                        outside[cuts[r]:cuts[r + 1]] = False
                        assert not part[outside].any()
                    acc[n] += part
        for n in range(len(modes)):
            e = np.linalg.norm(acc[n] - want[n]) / np.linalg.norm(want[n])
            assert e <= 1e-12, "sliced mode %d, output mode %d: %.3e" % (s, n, e)


@pytest.mark.gpu
def test_single_slab_run_equals_plain_run(pkg):
    import importlib
    import caseio
    from helpers import to_ktensors
    d = importlib.import_module("cp_cals_b200.distributed")
    rng = np.random.default_rng(77)
    modes = (20, 16, 30)
    X = rng.uniform(-1, 1, size=modes)
    ms = caseio.random_models(rng, modes, [4, 2, 7, 1])
    # a single slab that covers the whole tensor runs the very same kernels on the very same data, with and without the
    # pair node (cut along mode 2: T is local to the slab, csrc/pairnode.cuh); cut along mode 0 there is no pair node
    for method, s_mode, shared in (("mttkrp", 2, False), ("auto", 2, True), ("auto", 0, False)):
        p = pkg.CalsParams(max_iterations=6, buffer_size=14, force_max_iter=True, mttkrp_method=method)
        plain = to_ktensors(pkg, ms)
        rep0 = pkg.cp_cals(X, plain, pkg.CalsParams(max_iterations=6, buffer_size=14, force_max_iter=True,
                                                    mttkrp_method="auto" if shared else "mttkrp"))
        assert rep0.pair_node == shared
        sliced = to_ktensors(pkg, ms)
        rep = d.cp_cals_sliced(X, modes, s_mode, sliced, p)
        assert rep.iter == 6
        for a, b in zip(plain, sliced):
            assert all(np.array_equal(x, y) for x, y in zip(a.factors, b.factors)), (method, s_mode)
            assert np.array_equal(a.lam, b.lam) and a.error == b.error


@pytest.mark.gpu
def test_single_slab_run_forwards_update_method_and_line_search(pkg):
    """cp_cals_sliced honours CalsParams::update_method and line_search* exactly like cp_cals and the C++ run_sliced
    (ADVICE round 1: it used to run an unconstrained ALS without line search, silently)."""
    import importlib
    import caseio
    from helpers import to_ktensors
    d = importlib.import_module("cp_cals_b200.distributed")
    rng = np.random.default_rng(78)
    modes = (18, 14, 22)
    gen = [rng.uniform(0, 1, size=(i, 3)) for i in modes]
    X = caseio.ktensor_to_tensor(gen, np.ones(3)) + 0.02 * rng.uniform(0, 1, size=modes)
    ms = caseio.random_models(rng, modes, [3, 2, 5])
    for m in ms:
        m.factors = [np.abs(F) for F in m.factors]
    cases = [dict(update_method="nnls"),
             dict(line_search=True, line_search_interval=3, line_search_method="no-error-checking")]
    for extra in cases:
        p = pkg.CalsParams(max_iterations=7, buffer_size=10, force_max_iter=True, **extra)
        plain = to_ktensors(pkg, ms)
        rep0 = pkg.cp_cals(X, plain, p)
        sliced = to_ktensors(pkg, ms)
        rep = d.cp_cals_sliced(X, modes, 2, sliced, p)
        assert rep.iter == rep0.iter
        for a, b in zip(plain, sliced):
            assert all(np.array_equal(x, y) for x, y in zip(a.factors, b.factors)), extra
            assert np.array_equal(a.lam, b.lam) and a.error == b.error
        if "update_method" in extra:
            assert all((F >= 0).all() for k in sliced for F in k.factors)
            unconstrained = to_ktensors(pkg, ms)
            pkg.cp_cals(X, unconstrained, pkg.CalsParams(max_iterations=7, buffer_size=10, force_max_iter=True))
            assert any(not np.array_equal(a.factors[0], b.factors[0]) for a, b in zip(sliced, unconstrained))
    # the combination the sliced engine does not implement is refused, not emulated
    with pytest.raises(pkg.CalsB200Error):
        d.cp_cals_sliced(X, modes, 2, to_ktensors(pkg, ms),
                         pkg.CalsParams(max_iterations=3, buffer_size=10, update_method="nnls", line_search=True))


def _sliced_worker(rank, world, port, out_dir):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
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
        X, modes, ranks, ms = _sliced_case()
        for s in (2, 1, 0):  # 2, 1: pair node on every slab; 0: one MTTKRP per mode
            lo, hi = d.shard_slabs(modes[s], world)[rank]
            sl = [slice(None)] * len(modes)
            sl[s] = slice(lo, hi)
            kts = [pkg.Ktensor([F.copy() for F in m.factors]) for m in ms]
            rep = d.cp_cals_sliced(np.asfortranarray(X[tuple(sl)]), modes, s, kts,
                                   pkg.CalsParams(max_iterations=5, buffer_size=sum(ranks), force_max_iter=True),
                                   device=rank)
            np.savez(os.path.join(out_dir, "sliced_s%d_rank%d.npz" % (s, rank)), iter=rep.iter, x_norm=rep.X_norm,
                     **{"m%d_f%d" % (i, n): F for i, k in enumerate(kts) for n, F in enumerate(k.factors)},
                     **{"m%d_lam" % i: k.lam for i, k in enumerate(kts)},
                     **{"m%d_st" % i: np.array([k.iters, k.error, k.fit]) for i, k in enumerate(kts)})
    finally:
        dist.destroy_process_group()


def _sliced_case():
    import caseio
    rng = np.random.default_rng(5)
    modes = (26, 30, 44)
    X = rng.uniform(-1, 1, size=modes)
    ranks = [3, 6, 1, 12, 5]
    return X, modes, ranks, caseio.random_models(rng, modes, ranks)


@pytest.mark.gpu
def test_sliced_tensor_over_gpus_matches_oracle(tmp_path):
    """Real exchange over NVLink peer memory: W processes, one GPU each, X sliced along each of its modes in turn."""
    import torch
    import torch.multiprocessing as mp
    import oracle
    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    mp.spawn(_sliced_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    X, modes, ranks, ms = _sliced_case()
    want = oracle.cp_cals(X, ms, max_iter=5, force_max_iter=True)
    for s in (2, 1, 0):  # 2, 1: pair node on every slab; 0: one MTTKRP per mode
        outs = [np.load(os.path.join(str(tmp_path), "sliced_s%d_rank%d.npz" % (s, r))) for r in range(world)]
        for k in outs[0].files:  # replicated state: bit-identical on every GPU
            for o in outs[1:]:
                assert np.array_equal(outs[0][k], o[k]), k
        assert int(outs[0]["iter"]) == want.iters
        assert abs(float(outs[0]["x_norm"]) - want.x_norm) <= 1e-12 * want.x_norm
        for i, w in enumerate(want.models):
            for n in range(len(modes)):
                a = outs[0]["m%d_f%d" % (i, n)]
                assert np.linalg.norm(a - w.factors[n]) <= 1e-9 * np.linalg.norm(w.factors[n])
            assert np.linalg.norm(outs[0]["m%d_lam" % i] - w.lam) <= 1e-9 * np.linalg.norm(w.lam)
            st = outs[0]["m%d_st" % i]
            assert int(st[0]) == w.iters and abs(st[2] - w.fit) <= 1e-9
