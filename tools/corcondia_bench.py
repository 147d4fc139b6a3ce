"""Time the core consistency call (Engine.core_consistency, csrc/corcon.cuh) on BASELINE configs 2 and 4.

  python tools/corcondia_bench.py --out DIR [--reps 20]

Config 2: 200^3, 200 models (ranks 1..20, ten each), scored after a 50-iteration run (fitted factors).
Config 4: 80^4, 150 models (ranks 1..30, five each), scored as enqueued.
Per config: the call's device time (CUDA events on the engine stream, mean over --reps calls after a warm-up call), the
split between the shared contraction (pair_gemm_kernel) and the per-model kernels (corcon_*) from torch.profiler in a
separate call, the shared contraction's TFLOP/s against the 37.0 TFLOP/s DMMA peak, the time of two ALS iterations of
the same queue (config 2), and the host time of the NumPy reference on the same models for context.  The card's name and
power limit go with the numbers.  Results: DIR/corcondia_bench.json.
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import caseio  # noqa: E402
from test_core_consistency import corcondia_ref  # noqa: E402

DMMA_PEAK_TFLOPS = 37.0


def load_package():
    path = os.path.join(ROOT, "cp-cals_b200", "__init__.py")
    spec = importlib.util.spec_from_file_location("cp_cals_b200", path, submodule_search_locations=[os.path.dirname(path)])
    mod = importlib.util.module_from_spec(spec)
    sys.modules["cp_cals_b200"] = mod
    spec.loader.exec_module(mod)
    return mod


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def time_call(torch, eng, reps):
    stream = torch.cuda.ExternalStream(eng.stream_handle())
    eng.core_consistency()  # warm-up: workspace, module load
    t_host, ms = 0.0, []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        h0 = time.perf_counter()
        cc, st = eng.core_consistency()
        t_host += time.perf_counter() - h0
        e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return cc, st, float(np.mean(ms)), float(np.std(ms)), 1e3 * t_host / reps


def split(torch, eng):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.core_consistency()
        torch.cuda.synchronize()
    out = {"pair_gemm_ms": 0.0, "pinv_ms": 0.0, "chain_ms": 0.0, "final_ms": 0.0}
    for ev in prof.key_averages():
        t = ev.device_time_total / 1e3 if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1e3
        for key, name in (("pair_gemm_ms", "pair_gemm_kernel"), ("pinv_ms", "corcon_pinv_kernel"),
                          ("chain_ms", "corcon_chain_kernel"), ("final_ms", "corcon_final_kernel")):
            if name in ev.key:
                out[key] += t
    return out


def numpy_reference(X, models, subset):
    idx = list(range(0, len(models), max(1, len(models) // subset)))[:subset]
    t0 = time.perf_counter()
    for i in idx:
        fs, lam = models[i]
        corcondia_ref(X, fs, lam)
    t = time.perf_counter() - t0
    ranks = [models[i][0][0].shape[1] for i in range(len(models))]
    scale = sum(ranks) / sum(ranks[i] for i in idx)  # the tensor-sized contraction dominates: time ~ rank
    return {"models_timed": len(idx), "seconds_timed": t, "seconds_all_models_extrapolated": t * scale}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--ref-subset", type=int, default=20, help="models the NumPy reference is timed on, per config")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    import torch
    pkg = load_package()
    res = {"card": card(), "dmma_peak_tflops": DMMA_PEAK_TFLOPS}

    for cfg, modes, ranks, run_iters in (("config2", (200, 200, 200), [r for r in range(1, 21) for _ in range(10)], 50),
                                         ("config4", (80, 80, 80, 80), [r for r in range(1, 31) for _ in range(5)], 0)):
        rng = np.random.default_rng(0)
        X = rng.uniform(-1, 1, size=modes)
        ms = caseio.random_models(rng, modes, ranks)
        eng = pkg.Engine(0)
        eng.set_tensor(X)
        eng.configure(4200, max(run_iters, 1), 1e-7, force_max_iter=True)
        eng.clear_models()
        eng.enqueue_many([m.factors for m in ms])
        r = {"modes": modes, "models": len(ranks), "cols": sum(ranks)}
        if run_iters:
            rep = eng.run()
            r["als_iteration_ms"] = rep.device_ms / rep.iter
            r["two_als_iterations_ms"] = 2 * rep.device_ms / rep.iter
            fitted = [(fs, lam) for fs, lam, _ in eng.fetch_all()]
        else:
            fitted = [(m.factors, None) for m in ms]
        cc, st, mean_ms, sd_ms, host_ms = time_call(torch, eng, args.reps)
        r.update(call_ms=mean_ms, call_ms_sd=sd_ms, call_host_ms=host_ms, status_counts=np.bincount(st).tolist())
        r.update(split(torch, eng))
        nX = float(np.prod(modes))
        r["shared_contraction_gflop"] = 2 * nX * sum(ranks) / 1e9
        r["shared_contraction_tflops"] = r["shared_contraction_gflop"] / r["pair_gemm_ms"] if r["pair_gemm_ms"] else None
        r["shared_contraction_share_of_peak"] = (r["shared_contraction_tflops"] or 0) / DMMA_PEAK_TFLOPS
        r["numpy_reference"] = numpy_reference(X, fitted, args.ref_subset)
        # spot check against the reference
        i = len(ranks) // 2
        r["spot_check"] = {"model": i, "device": float(cc[i]), "numpy": corcondia_ref(X, fitted[i][0], fitted[i][1])}
        eng.close()
        res[cfg] = r
        print(cfg, json.dumps(r, default=float))
    with open(os.path.join(args.out, "corcondia_bench.json"), "w") as fh:
        json.dump(res, fh, indent=1, default=float)
    print("card:", res["card"])


if __name__ == "__main__":
    main()
