"""Per-kernel split of one config-2 run under both schedules (run on the GPU box; torch.profiler with CUDA activities).

The multi-sweep schedule launches pair_gemm_kernel for nodes 2, 1 (even iteration) and 0 (odd iteration) in that order,
so the i-th launch of a run belongs to node (2, 1, 0)[i % 3]; the one-sweep schedule launches node 0 only.  Prints the
mean time per launch of every contraction kernel, per node, and of the leaf / reduce kernels.
Usage: python tools/msdt_nodes.py [config] [output dir (also writes config<N>.json there)]"""
import collections
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
from conftest import load_package  # noqa: E402

pkg = load_package()
cfg_id = int(sys.argv[1]) if len(sys.argv) > 1 else 2
out_dir = sys.argv[2] if len(sys.argv) > 2 else None
cfg = bench.CONFIGS[cfg_id]
X, models, jk = bench.workload(cfg, 0)
C = sum(fs[0].shape[1] for fs in models)
result = {"config": cfg_id, "columns": C}
for msdt in ("0", "1"):
    os.environ["CALS_B200_MSDT"] = msdt
    with pkg.Engine(0) as eng:
        eng.set_tensor(X)
        eng.configure(C, cfg["als_iters"], 1e-7, force_max_iter=True)
        eng.clear_models()
        eng.enqueue_many(models, jk)
        eng.run()  # allocations, graphs, warm-up
        eng.rerun()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            rep = eng.rerun()
        torch.cuda.synchronize()
    kern = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                  key=lambda e: e.time_range.start)
    per = collections.defaultdict(list)
    i_gemm = 0
    for e in kern:
        name = e.name.split("<")[0].replace("void ", "").replace("calsb200::", "")
        if name.startswith("pair_gemm_kernel") and msdt == "1":
            name += " node %d" % (2, 1, 0)[i_gemm % 3]
            i_gemm += 1
        per[name].append(e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total)
    iters = rep.iter
    result["msdt=" + msdt] = {
        "iterations": iters, "sweep_period": rep.sweep_period, "device_ms_per_iteration": rep.device_ms / iters,
        "kernels": {k: {"launches": len(v), "us_per_launch": sum(v) / len(v), "us_per_iteration": sum(v) / iters}
                    for k, v in sorted(per.items())}}
txt = json.dumps(result, indent=1)
if out_dir:
    os.makedirs(out_dir, exist_ok=True)
    open(os.path.join(out_dir, "config%d.json" % cfg_id), "w").write(txt)
print(txt)
