"""Cost of models above the shared-memory update kernel's rank bound (the wide path, csrc/wide.cuh) next to config 2.

One seeded 200^3 tensor, forced iterations, four queues timed in the same process, alternating:
  (a) config 2's model set: ranks 1..20 x10, 2100 columns
  (b) 8 models of rank 256: 2048 columns
  (c) 2 models of rank 1024
  (d) config 2's models plus 4 of rank 128
For each: seconds per global iteration and model-iterations/s (untimed runs), and mttkrp_ms / update_ms per iteration
from a run with per-kernel timing.  The card's name and power limit are read in the same call.
Usage: python tools/wide_rank_bench.py [--iters K] [--rounds N] [--out DIR]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from __graft_entry__ import load_package  # noqa: E402

QUEUES = {
    "a": [r for r in range(1, 21) for _ in range(10)],
    "b": [256] * 8,
    "c": [1024] * 2,
    "d": [r for r in range(1, 21) for _ in range(10)] + [128] * 4,
}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    pkg = load_package()
    rng = np.random.default_rng(0)
    modes = (200, 200, 200)
    X = rng.uniform(-1, 1, size=modes)
    models = {}
    for k, ranks in QUEUES.items():
        models[k] = [[rng.uniform(-1, 1, size=(i, r)) for i in modes] for r in ranks]
    res = {k: {"ranks": "%d models, %d columns" % (len(v), sum(v)), "s_per_iteration": []} for k, v in QUEUES.items()}
    with pkg.Engine(0) as eng:
        eng.set_tensor(X)
        for rnd in range(args.rounds + 1):  # round 0 warms every queue up (allocations, graphs)
            for k, ranks in QUEUES.items():
                eng.configure(sum(ranks), args.iters, 1e-7, force_max_iter=True)
                eng.clear_models()
                eng.enqueue_many(models[k])
                eng.run()
                t0 = time.perf_counter()
                rep = eng.rerun()
                dt = time.perf_counter() - t0
                if rnd > 0:
                    res[k]["s_per_iteration"].append(rep.device_ms / 1e3 / rep.iter)
                if rnd == args.rounds:  # one timing run per queue
                    eng.set_timing(1)
                    t = eng.rerun()
                    eng.set_timing(0)
                    res[k]["mttkrp_ms_per_iteration"] = t.mttkrp_ms / t.iter
                    res[k]["update_ms_per_iteration"] = t.update_ms / t.iter
                    res[k]["host_s_last_run"] = dt
    for k, ranks in QUEUES.items():
        s = float(np.median(res[k]["s_per_iteration"]))
        res[k]["median_s_per_iteration"] = s
        res[k]["model_iterations_per_s"] = len(ranks) / s
    out = {"card": card(), "tensor": "200x200x200", "forced_iterations": args.iters, "queues": res,
           "b_over_a": res["b"]["median_s_per_iteration"] / res["a"]["median_s_per_iteration"]}
    txt = json.dumps(out, indent=1)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "wide_rank_bench.json"), "w") as f:
            f.write(txt)
    print(txt)


if __name__ == "__main__":
    main()
