#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 CP-CALS hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1|2|3|4|5]
                    [--weak] [--no-secondary] [--no-cpu-baseline] [--dump-outputs DIR]

Metric (BASELINE.json): concurrent-ALS iterations per second summed over all models ("model-iterations/s").  The
headline workload is BASELINE config 2 (the largest configuration the metric is quoted on that fits one GPU): synthetic
200x200x200 FP64 tensor, 200 concurrent models (ranks 1..20 x 10), buffer = sum of ranks, forced iteration count.
One "step" = one complete cals::cp_cals pass: all 200 models x 50 forced ALS iterations (the iteration count of the
reference's own experiments, src/experiments/experiments.cpp:62-63).

  value    : whole-job throughput with the tensor and the initial models already resident in HBM (cals_b200_rerun),
             timed with CUDA events on the engine's stream, max over ranks
  e2e      : same metric through the drop-in C++ API -- cals::cp_cals of libcals.so over HOST containers (the program
             examples/bench_e2e.cpp): H2D of X and of the initial models, the loop, and D2H of every fitted model inside
             the timed region; `e2e.python` is the same through the ctypes wrapper
  roofline : the tensor-core contractions (dominant), algorithmic 2*nX*C flop per launch / CUDA-event time per launch,
             against the measured FP64 DMMA peak of this pool's B200 (profiles/fp64_peak_r01.json; MEASURED_PEAKS.json
             has no FP64 entry); `traffic` from the ncu capture profiles/traffic_r02.json, used only while its kernel
             fingerprint equals that of the sources this run was built from
  parity   : the GPU arm against the UNMODIFIED reference (oracle/_ref) on this very workload after a few forced
             iterations: largest relative error over every factor matrix, lambda and fit of all models
  cpu_baseline : the unmodified reference timed on the box's host cores on a bounded sample
  secondary    : the other BASELINE configurations at the same GPU count, each with its own clocks / roofline / e2e

--dump-outputs DIR writes the fitted models of the last timed step of the headline run as float64 .npy files, so that
two builds can be compared output for output: the inputs are seeded and identical from run to run.  On N > 1 GPUs only
rank 0 writes, and what it writes is its own share: the models shard_models assigns to rank 0 (strong scaling), or
rank 0's own model set (--weak); the sliced config 5 replicates the models, so there it is the whole set.

N > 1 (torchrun): the tensor is replicated and ONE model set (for the jackknife: one set of leave-one-out sub-models) is
sharded over the ranks -- strong scaling, no collective on the data path (north_star's partition; SURVEY 8e).  `--weak`
gives every rank its own full model set instead.  Config 5 slices the tensor over the ranks.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "concurrent-ALS iters/sec (all models)"
UNIT = "model-iterations/s"
RTOL = 1e-9  # north_star: per-iteration fit and factor matrices within 1e-9 relative error

# BASELINE.json configs.  als_iters: forced ALS iterations per model per step (config 2: 50, the protocol of the
# reference's own experiments, src/experiments/experiments.cpp:62-63); ref_iters: per step of the CPU reference (a bounded
# sample: the reference's one-off setup is reported separately so that the two arms can be compared per iteration).
CONFIGS = {
    1: dict(name="config 1: 100x100x100 tensor, 40 models (ranks 1..10 x4), buffer 220", modes=(100, 100, 100),
            ranks=[r for r in range(1, 11) for _ in range(4)], als_iters=50, ref_iters=20, jk=False),
    2: dict(name="config 2: 200x200x200 tensor, 200 models (ranks 1..20 x10), buffer 2100", modes=(200, 200, 200),
            ranks=[r for r in range(1, 21) for _ in range(10)], als_iters=50, ref_iters=10, jk=False),
    3: dict(name="config 3: jackknife on a 299x301x41 tensor (fluorescence_cancer_UD shape, synthetic), all 299 "
                 "leave-one-out sub-models of base models of ranks 3,5,7,9", modes=(299, 301, 41),
            ranks=[r for r in (3, 5, 7, 9) for _ in range(299)], als_iters=10, ref_iters=2, jk=True),
    4: dict(name="config 4: 80x80x80x80 tensor, 150 models (ranks 1..30 x5), buffer 2325", modes=(80, 80, 80, 80),
            ranks=[r for r in range(1, 31) for _ in range(5)], als_iters=4, ref_iters=1, jk=False),
    5: dict(name="config 5: 1000x1000x1000 tensor sliced along mode 2 over the GPUs, 50 models (ranks 1..50), buffer "
                 "1275, partial MTTKRPs combined over NVLink peer memory", modes=(1000, 1000, 1000),
            ranks=list(range(1, 51)), als_iters=2, ref_iters=1, jk=False, sliced=2),
}


def init_nccl(local_rank):
    """init_process_group + the first collective (which creates the communicator) with file descriptor 1 pointed at
    stderr: NCCL prints its version banner on STDOUT at that moment, and stdout is reserved for the one JSON line."""
    import torch
    import torch.distributed as dist
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
        torch.cuda.synchronize()
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)
    return dist


def load_pkg():
    from conftest import load_package
    return load_package()


def workload(cfg, seed):
    """Synthetic inputs as the reference driver makes them (src/examples/driver.cpp:133-153): X uniform(-1,1), models
    uniform(-1,1) then Ktensor::normalize().  X is the same on every rank (replicated); models differ with `seed`.
    Jackknife config: sub-model i of a base model is that model flagged "leave mode-0 sample i out" (the reference
    derives them from fitted base models; for throughput the starting values do not matter)."""
    modes = cfg["modes"]
    rng = np.random.default_rng(1234)
    X = np.asfortranarray(rng.uniform(-1.0, 1.0, size=modes))
    mrng = np.random.default_rng(1000 + seed)
    models, jk = [], []
    base = {}
    for idx, r in enumerate(cfg["ranks"]):
        if cfg["jk"] and r in base:
            fs = base[r]
        else:
            fs = []
            for i in modes:
                F = mrng.uniform(-1.0, 1.0, size=(i, r))
                fs.append(np.asfortranarray(F / np.linalg.norm(F, axis=0)))
            base[r] = fs
        models.append(fs)
        jk.append((0, idx % modes[0]) if cfg["jk"] else (-1, 0))
    return X, models, jk


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms.  Started BEFORE the warm-up of a run (nvidia-smi takes
    a few hundred ms to deliver its first line, longer than the timed region of the small configurations); only samples
    taken while the SMs were clocked up (> half of the maximum) count as "under load"."""
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def wait_first_sample(self, timeout=3.0):
        t0 = time.perf_counter()
        while self.proc and not self.lines and time.perf_counter() - t0 < timeout:
            time.sleep(0.02)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        busy = [s for s in sm if mx and s > 0.5 * mx] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "samples_under_load": len(busy) if busy is not sm else 0}


def fp64_peak():
    path = os.path.join(ROOT, "profiles", "fp64_peak_r01.json")
    try:
        with open(path) as f:
            d = json.load(f)
        return float(d["dmma_tflops_sustained"]), "measured (tools/fp64_peak.cu, profiles/fp64_peak_r01.json)"
    except Exception:
        return 37.0, "fallback (no profiles/fp64_peak_r01.json)"


def measured_hbm_peak():
    """HBM copy bandwidth of this pool's B200 in GB/s: MEASURED_PEAKS.json (driver-written), else the profiling
    recipe's fallback."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"])
    except Exception:
        return 6534.8


def kernel_fingerprint():
    """SHA-256 over the kernel sources the product library is built from (cp-cals_b200/csrc) and its Makefile: the
    identity of the code an ncu capture describes.  tools/ncu_summary.py stamps it into profiles/traffic_r02.json."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "cp-cals_b200", "csrc")
    for name in sorted(os.listdir(d)) + ["../Makefile"]:
        with open(os.path.join(d, name), "rb") as f:
            h.update(name.encode() + b"\0" + f.read())
    return h.hexdigest()[:16]


def stored_traffic(kernel_prefix, workload_key):
    """DRAM bytes per launch of a kernel from the committed ncu capture -- only if that capture was taken on the code
    this run uses.  Returns (bytes or None, note)."""
    path = os.path.join(ROOT, "profiles", "traffic_r02.json")
    try:
        with open(path) as f:
            d = json.load(f)
    except Exception:
        return None, "no profiles/traffic_r02.json (tools/refresh_traffic.sh makes it)"
    now = kernel_fingerprint()
    if d.get("kernel_fingerprint") != now:
        return None, ("profiles/traffic_r02.json describes kernel sources %s, this run was built from %s: refused as "
                      "stale (re-run tools/refresh_traffic.sh)" % (d.get("kernel_fingerprint"), now))
    for e in d.get("kernels", []):
        if e["kernel"].startswith(kernel_prefix) and e.get("workload") == workload_key:
            return float(e["dram_bytes_per_launch"]), "ncu --set full, %s, sources %s" % (d.get("captured", "?"), now)
    return None, "profiles/traffic_r02.json has no entry for %s on %s" % (kernel_prefix, workload_key)


# ---------------------------------------------------------------------------------------------------------------------
# CPU reference legs (oracle/ is test infrastructure: allowed here as the CPU baseline / reference arm / parity checker)
def _caseio():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import caseio
    return caseio


def _ref_models(caseio, models, jk):
    return [caseio.Model(factors=fs, jk_mode=j[0], jk_fiber=j[1]) for fs, j in zip(models, jk)]


def run_reference_sample(X, models, jk, iters, threads, release=True):
    """One cals::cp_cals call of the unmodified reference; returns its RefResult (seconds = the reference's own
    total_time: setup -- ||X||, workspaces, initial Gramians -- plus `iters` iterations)."""
    caseio = _caseio()
    ms = _ref_models(caseio, models, jk)
    return caseio.run_reference(X, ms, max_iter=iters, force_max_iter=True, threads=threads, release=release,
                                buffer_size=sum(m.rank for m in ms))


def reference_rate(X, models, jk, iters, threads):
    """Times the reference at 1 and at `iters` forced iterations and separates its one-off setup from the per-iteration
    cost: t(k) = setup + k * per_iter.  Returns a dict."""
    t1 = run_reference_sample(X, models, jk, 1, threads).seconds
    tk = run_reference_sample(X, models, jk, iters, threads).seconds
    per_iter = max((tk - t1) / max(iters - 1, 1), 1e-9) if iters > 1 else t1
    setup = max(t1 - per_iter, 0.0) if iters > 1 else 0.0
    return {"seconds": tk, "iters": iters, "setup_s": setup, "per_iteration_s": per_iter,
            "value": len(models) * iters / tk, "marginal_value": len(models) / per_iter}


def cpu_baseline(cfg, X, models, jk):
    caseio = _caseio()
    if not caseio.ref_available():
        return {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "oracle/_ref not built"}
    iters = cfg["ref_iters"]
    ncpu = os.cpu_count() or 1
    r = reference_rate(X, models, jk, iters, ncpu)
    proj = len(models) * cfg["als_iters"] / (r["setup_s"] + cfg["als_iters"] * r["per_iteration_s"])
    return {"value": r["value"], "unit": UNIT, "cores": ncpu, "kind": "reference",
            "setup_s": r["setup_s"], "per_iteration_s": r["per_iteration_s"], "marginal_value": r["marginal_value"],
            "projected_value_at_gpu_arm_iters": proj,
            "binary": os.path.basename(caseio.ref_binary(True)),
            "sample": "unmodified reference cp_cals (OpenBLAS, the reference's Release flags -O3 -ffast-math), full model "
                      "set of the workload, %d forced ALS iterations in %.2f s of cp_cals time, %d threads "
                      "(OMP_WAIT_POLICY=passive); a 1-iteration run beside it separates the one-off setup (%.2f s) from "
                      "the per-iteration cost (%.3f s): marginal_value is the rate without setup, "
                      "projected_value_at_gpu_arm_iters the rate the reference would reach at the GPU arm's %d "
                      "iterations per step" % (iters, r["seconds"], ncpu, r["setup_s"], r["per_iteration_s"],
                                               cfg["als_iters"])}


def parity_check(pkg, eng, cfg, X, models, jk, iters=2):
    """GPU arm vs the unmodified reference (plain, no-fast-math build) on the bench workload itself: same inputs, same
    forced iteration count, every model.  Returns the `parity` object of the JSON line."""
    caseio = _caseio()
    if not caseio.ref_available():
        return {"max_rel_err": None, "note": "oracle/_ref not built"}
    C = sum(fs[0].shape[1] for fs in models)
    ref = caseio.run_reference(X, _ref_models(caseio, models, jk), max_iter=iters, force_max_iter=True,
                               threads=os.cpu_count() or 1, buffer_size=C)
    kts = [pkg.Ktensor([np.array(F, order="F", copy=True) for F in fs], None, j[0], j[1]) for fs, j in zip(models, jk)]
    pkg.cp_cals(X, kts, pkg.CalsParams(max_iterations=iters, buffer_size=C, force_max_iter=True), engine=eng)
    worst = {"factor": 0.0, "lambda": 0.0, "fit": 0.0}
    for g, r in zip(kts, ref.models):
        for Fg, Fr in zip(g.factors, r.factors):
            worst["factor"] = max(worst["factor"], float(np.linalg.norm(Fg - Fr) / np.linalg.norm(Fr)))
        worst["lambda"] = max(worst["lambda"], float(np.linalg.norm(g.lam - r.lam) / np.linalg.norm(r.lam)))
        worst["fit"] = max(worst["fit"], abs(g.fit - (1.0 - abs(r.error) / ref.x_norm)))
    mx = max(worst.values())
    return {"max_rel_err": mx, "factor": worst["factor"], "lambda": worst["lambda"], "fit_abs": worst["fit"],
            "iters": iters, "models": len(models), "tolerance": RTOL, "ok": bool(mx <= RTOL),
            "against": "unmodified reference cals::cp_cals (oracle/_ref/cals_ref, no -ffast-math), same inputs, %d "
                       "forced iterations, all %d models" % (iters, len(models))}


def reference_arm(args, cfg, rank):
    if rank != 0:
        return
    X, models, jk = workload(cfg, 0)
    ncpu = os.cpu_count() or 1
    warm = args.warmup if args.warmup is not None else 1
    it = cfg["ref_iters"]
    t1 = None
    for _ in range(warm):  # warm-up steps double as the 1-iteration runs that isolate the reference's setup time
        t1 = run_reference_sample(X, models, jk, 1, ncpu).seconds
    steps = args.steps if args.steps is not None else 3
    secs = [run_reference_sample(X, models, jk, it, ncpu).seconds for _ in range(steps)]
    t = float(np.mean(secs))
    v = len(models) * it / t
    extra = {}
    if t1 is not None and it > 1:
        per_iter = max((t - t1) / (it - 1), 1e-9)
        setup = max(t1 - per_iter, 0.0)
        extra = {"setup_s": setup, "per_iteration_s": per_iter, "marginal_value": len(models) / per_iter,
                 "projected_value_at_gpu_arm_iters":
                     len(models) * cfg["als_iters"] / (setup + cfg["als_iters"] * per_iter)}
    caseio = _caseio()
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": 0, "steps": steps,
            "warmup": warm, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": cfg["name"], "als_iters_per_step": it, "l2": "inputs larger than L2",
                       "same_config": "same tensor, same %d models, same buffer as the GPU arm at every GPU count (the "
                                      "GPU arm shards this one model set); the GPU arm runs %d forced iterations per "
                                      "step, this arm %d (bounded sample) with the reference's one-off setup inside "
                                      "every step -- setup_s / per_iteration_s / projected_value_at_gpu_arm_iters in "
                                      "cpu_baseline give the like-for-like rate" % (len(models), cfg["als_iters"], it)},
            "cpu_baseline": dict({"value": v, "unit": UNIT, "cores": ncpu, "kind": "reference",
                                  "binary": os.path.basename(caseio.ref_binary(True)),
                                  "sample": "each step = %d forced ALS iterations of the full model set through the "
                                            "unmodified reference's cp_cals (its own total_time), built with the "
                                            "reference's Release flags, %d threads" % (it, ncpu)}, **extra),
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
class Dist:
    """barrier / max / min over ranks; no-ops on one GPU."""

    def __init__(self, dist):
        self.dist = dist

    def barrier(self):
        import torch
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def _reduce(self, x, op):
        if self.dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max(self, x):
        return self._reduce(x, self.dist.ReduceOp.MAX) if self.dist is not None else x

    def min(self, x):
        return self._reduce(x, self.dist.ReduceOp.MIN) if self.dist is not None else x

    def sum(self, x):
        return self._reduce(x, self.dist.ReduceOp.SUM) if self.dist is not None else x


def dump_outputs(eng, out_dir):
    """The models of the engine's last run as a caller of cp_cals receives them: per mode the factor matrices of all
    models side by side (I_n x sum of ranks, queue order), lambda, and per model the iteration count, error and fit.
    Every file is float64; the largest configuration (config 3) comes to about 37 MB."""
    os.makedirs(out_dir, exist_ok=True)
    res = eng.fetch_all()
    arrays = {"lambda": np.concatenate([lam for _, lam, _ in res])}
    for n in range(len(eng.modes)):
        arrays["factors_mode%d" % n] = np.concatenate([fs[n] for fs, _, _ in res], axis=1)
    for key in ("iters", "error", "fit"):
        arrays[key] = np.array([getattr(st, key) for _, _, st in res])
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def cpp_e2e(cfg, X, models, jk, als_iters, steps, warmup, device, no_pair_node=False, nnls=False):
    """The end-to-end leg through the drop-in C++ API: examples/bench_e2e.cpp (cals::cp_cals of libcals.so) on a case
    file holding exactly these inputs.  Returns its JSON dict, or None when the program is missing / failed."""
    exe = os.path.join(ROOT, "cp-cals_b200", "bin", "bench_e2e")
    if not os.path.exists(exe):
        return None
    caseio = _caseio()
    ms = _ref_models(caseio, models, jk)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "case.in")
        caseio.write_case(path, X, ms, max_iter=als_iters, force_max_iter=True, buffer_size=sum(m.rank for m in ms),
                          mttkrp_method=caseio.METHOD_MTTKRP if no_pair_node else caseio.METHOD_AUTO, nnls=nnls)
        p = subprocess.run([exe, path, str(steps), str(warmup), str(device)], capture_output=True, text=True,
                           timeout=1200)
    if p.returncode != 0:
        sys.stderr.write("bench_e2e failed (%d): %s\n" % (p.returncode, p.stderr[-1000:]))
        return None
    for ln in p.stdout.splitlines():
        if ln.startswith("{"):
            return json.loads(ln)
    return None


def run_sharded(args, cfg_id, rank, world, local_rank, D, steps, warmup, main_line, dump_dir=None):
    """Configs 1-4: tensor replicated, model set sharded over the ranks.  Returns the line (rank 0) or None."""
    import importlib

    import torch
    cfg = CONFIGS[cfg_id]
    als_iters = cfg["als_iters"]
    sampler = ClockSampler(local_rank).start()
    pkg = load_pkg()
    dmod = importlib.import_module("cp_cals_b200.distributed")
    strong = not args.weak
    X, models, jk = workload(cfg, 0 if strong else rank)
    all_models, all_jk = models, jk
    total_models = len(models) if strong else world * len(models)
    if strong and world > 1:
        mine = dmod.shard_models([fs[0].shape[1] for fs in models], world)[rank]
        models, jk = [models[i] for i in mine], [jk[i] for i in mine]
    if args.shard_of > 1 and world == 1:
        mine = dmod.shard_models([fs[0].shape[1] for fs in models], args.shard_of)[0]
        models, jk = [models[i] for i in mine], [jk[i] for i in mine]
        all_models, all_jk = models, jk
        total_models = len(models)
    nX = X.size
    modes = X.shape
    C = sum(fs[0].shape[1] for fs in models)
    n_models = len(models)

    eng = pkg.Engine(local_rank)
    eng.set_tensor(X)
    eng.configure(C, als_iters, 1e-7, force_max_iter=True, nnls=args.nnls)
    eng.set_pair_node(not args.no_pair_node)
    eng.clear_models()
    for fs, j in zip(models, jk):
        eng.enqueue(fs, j[0], j[1])
    eng.run()  # uploads + first pass (untimed)
    # CUDA events are recorded on the stream the engine launches on (torch's current stream would see nothing)
    es = torch.cuda.ExternalStream(eng.stream_handle(), device=torch.device("cuda", local_rank))

    def timed(fn, n):
        """n calls of fn bracketed by barrier + synchronize; returns (device ms between events, wall seconds)."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        D.barrier()
        t0 = time.perf_counter()
        ev0.record(es)
        out = [fn() for _ in range(n)]
        ev1.record(es)
        D.barrier()
        t1 = time.perf_counter()
        return ev0.elapsed_time(ev1), t1 - t0, out

    # ---------------- value: inputs resident ----------------
    sampler.wait_first_sample()
    t_w = time.perf_counter()
    done_w = 0
    while done_w < warmup or (time.perf_counter() - t_w < 0.4 and done_w < 400):  # at least W steps and 0.4 s under load
        eng.rerun()
        done_w += 1
    done_w = int(D.max(done_w))
    ev_ms, wall, reps = timed(eng.rerun, steps)
    clocks = sampler.stop()
    if dump_dir and rank == 0:
        dump_outputs(eng, dump_dir)
    launches = sum(r.kernel_launches for r in reps)
    assert all(r.iter == als_iters and r.n_ktensors == n_models for r in reps)
    ev_ms = D.max(ev_ms)       # CUDA events on the engine stream around the K steps, max over ranks
    wall = D.max(wall)         # host clock around the same region (reported beside it)
    value = total_models * als_iters * steps / (ev_ms * 1e-3)

    # ---------------- roofline of the dominant kernel (extra passes with per-kernel CUDA events) ----------------
    eng.set_timing(1)
    mt_ms, mt_launches, up_ms, gemm_ms, leaf_ms, tensor_flops, tree = 0.0, 0, 0.0, 0.0, 0.0, 0.0, False
    fused_blocks = 0
    for _ in range(2):
        rep = eng.rerun()
        fused_blocks = int(rep.fused_leaf_blocks)
        mt_ms += rep.mttkrp_ms
        up_ms += rep.update_ms
        mt_launches += rep.mttkrp_launches
        gemm_ms += rep.pair_gemm_ms
        leaf_ms += rep.pair_leaf_ms
        tensor_flops += rep.tensor_flops
        tree = tree or bool(rep.tree)
    eng.set_timing(0)
    # The tensor-core kernels: one full MTTKRP per mode, or -- pair nodes (csrc/pairnode.cuh) -- the MTTKRP of mode 0 and
    # the shared contraction T = X_(0)^T A_0 (3 modes) / two pair contractions (4 modes); each launch is one
    # tensor-sized contraction of 2*nX*C flop.
    flops_per_launch = 2.0 * nX * C
    tensor_ms = mt_ms - leaf_ms
    tensor_launches = tensor_flops / flops_per_launch
    ach_local = tensor_flops / (tensor_ms * 1e-3) / 1e12
    ach = D.min(ach_local)  # the slowest GPU's rate
    peak, peak_src = fp64_peak()
    iters_timed = mt_launches / len(modes)  # ALS iterations covered by the per-kernel timing passes
    step_ms_per_iter = ev_ms / steps / als_iters
    shares = {"tensor_contractions": D.max(tensor_ms / iters_timed) / step_ms_per_iter,
              "pair_leaves_hbm": D.max(leaf_ms / iters_timed) / step_ms_per_iter,
              "per_model_update": D.max(up_ms / iters_timed) / step_ms_per_iter}
    shares["scheduler_moves_and_launch_gaps"] = max(0.0, 1.0 - sum(shares.values()))
    traffic, traffic_note = (None, "not captured for this configuration")
    if cfg_id == 2 and world == 1 and not args.no_pair_node and not args.shard_of:
        traffic, traffic_note = stored_traffic("mttkrp_dmma_kernel", "config2")
    roofline = {"bound": "tensor",
                "kernel": "mttkrp_dmma_kernel (timed together with its mttkrp_reduce_kernel)" +
                          (" and the pair-node contraction (pair_gemm_kernel)" if tree and len(modes) == 3 else ""),
                "achieved": ach, "peak": peak, "unit": "TFLOP/s" if world == 1 else "TFLOP/s per GPU (slowest rank)",
                "frac": ach / peak, "traffic": traffic, "traffic_source": traffic_note, "peak_source": peak_src,
                "ms_per_launch": D.max(tensor_ms / tensor_launches), "flops_per_launch": flops_per_launch,
                "columns_on_this_gpu": C,
                "launches_per_als_iteration": tensor_launches / iters_timed,
                "flop_count": "algorithmic 2*nX*C per tensor-sized contraction actually executed; the pair nodes run "
                              "%d of the reference's %d contractions per ALS iteration, so in SURVEY 8(d)'s count "
                              "(2*N*nX*C per iteration) the step rate is algorithmic_mttkrp_tflops, which may exceed "
                              "the DMMA peak" % (round(tensor_launches / iters_timed), len(modes)),
                "mttkrp_ms_per_mode": mt_ms / mt_launches,
                "share_of_step": shares,
                "limiter": max(shares, key=shares.get)}
    if tree:
        iters = iters_timed
        # 3 modes: one pair node (modes 1, 2) next to the full MTTKRP of mode 0; 4 modes: two pair nodes (0, 1), (2, 3)
        node_rows = [modes[1] * modes[2]] if len(modes) == 3 else [modes[0] * modes[1], modes[2] * modes[3]]
        full_modes = len(modes) - 2 * len(node_rows)
        leaf_launches = 2 * len(node_rows) * iters
        if fused_blocks:
            # 3 modes, first leaf in the contraction's epilogue: its pass reads fused_blocks partial results per element
            # of G_1 (I1 x C) instead of T; the second leaf streams T once
            leaf_bytes = (8.0 * node_rows[0] * C + 8.0 * fused_blocks * modes[1] * C) * iters
        else:
            leaf_bytes = sum(2 * 8.0 * r * C for r in node_rows) * iters  # every leaf streams its node's T once
        pn = {
            "what": "two modes take their MTTKRP from one shared contraction T (csrc/pairnode.cuh): %d tensor-sized "
                    "contractions per ALS iteration instead of %d; the leaf kernels stream T from HBM"
                    % (full_modes + len(node_rows), len(modes)) +
                    ("; the first leaf rides in the contraction's epilogue (its launch sums %d per-tile partial results "
                     "per element), so T is read once per iteration and pair_contraction_tflops includes that work"
                     % fused_blocks if fused_blocks else ""),
            "first_leaf_fused": bool(fused_blocks),
            "mttkrp_dmma_ms_per_launch": (tensor_ms - gemm_ms) / (iters * full_modes) if full_modes else None,
            "pair_contraction_ms_per_launch": gemm_ms / (iters * len(node_rows)),
            "pair_contraction_tflops": flops_per_launch / (gemm_ms / (iters * len(node_rows)) * 1e-3) / 1e12,
            "leaf_ms_per_launch": leaf_ms / leaf_launches if leaf_ms > 0 else None,
            "leaf_bytes_per_launch": leaf_bytes / leaf_launches,
            "leaf_achieved_gbs": leaf_bytes / (leaf_ms * 1e-3) / 1e9 if leaf_ms > 0 else None,
            "leaf_peak_gbs": measured_hbm_peak(),
            "algorithmic_mttkrp_tflops": len(modes) * flops_per_launch * iters / (mt_ms * 1e-3) / 1e12,
        }
        if traffic is not None:
            pn["pair_contraction_traffic"] = stored_traffic("pair_gemm_kernel", "config2")[0]
        roofline["pair_node"] = pn

    # ---------------- e2e: public API, host buffers in pinned memory ----------------
    def pinned_copy(a):
        t = torch.empty(a.size, dtype=torch.float64, pin_memory=True)
        v = t.numpy().reshape(a.shape, order="F")
        v[...] = a
        return t, v

    keep = []
    tX, Xp = pinned_copy(X)
    keep.append(tX)
    pinned_models = []
    for fs in models:
        row = []
        for F in fs:
            t, v = pinned_copy(F)
            keep.append(t)
            row.append(v)
        pinned_models.append(row)
    params = pkg.CalsParams(max_iterations=als_iters, buffer_size=C, force_max_iter=True,
                            update_method="nnls" if args.nnls else "unconstrained",
                            mttkrp_method="mttkrp" if args.no_pair_node else "auto")
    h2d = X.nbytes + sum(F.nbytes for fs in models for F in fs)
    d2h = sum(F.nbytes for fs in models for F in fs) + 8 * C + n_models * 40

    def e2e_step():
        kts = [pkg.Ktensor(list(fs), None, j[0], j[1]) for fs, j in zip(pinned_models, jk)]
        rep = pkg.cp_cals(Xp, kts, params, engine=eng)
        return rep, kts

    e2e_steps = max(2, min(steps, 5))
    e2e_step()
    e2e_ms, e2e_wall, outs = timed(e2e_step, e2e_steps)
    rep, kts = outs[-1]
    e2e_ms = D.max(e2e_ms)
    e2e_wall = D.max(e2e_wall)
    # the end-to-end step includes host work (queue packing, result unpacking) that no CUDA event sees once the
    # stream is idle, so the slower of the two clocks is the honest one
    e2e_t = max(e2e_ms * 1e-3, e2e_wall)
    py_e2e = {"value": total_models * als_iters * e2e_steps / e2e_t, "ms_per_step": e2e_t / e2e_steps * 1e3,
              "api": "cp_cals of the ctypes wrapper (cp-cals_b200/__init__.py), warm engine"}
    fit_checksum = float(np.mean([k.fit for k in kts]))

    # parity of this very workload against the unmodified reference (rank 0, one GPU, main line only)
    parity = None
    if main_line and rank == 0 and world == 1 and not args.no_cpu_baseline and not args.nnls:
        try:
            parity = parity_check(pkg, eng, cfg, X, models, jk)
        except Exception as e:
            parity = {"max_rel_err": None, "note": "failed: %s" % e}
    eng.close()
    del eng

    # the same through the drop-in C++ API (its own process per rank, after this process has released its engine)
    cpp = None
    try:
        cpp = cpp_e2e(cfg, X, models, jk, als_iters, e2e_steps, 2, local_rank, args.no_pair_node, args.nnls)
    except Exception as e:
        sys.stderr.write("bench_e2e: %s\n" % e)
    cpp_s = D.max(cpp["s_per_step"] if cpp else -1.0)
    cpp_ok = D.min(1.0 if cpp else 0.0) > 0.5
    if cpp_ok:
        e2e = {"value": total_models * als_iters / cpp_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "steps": e2e_steps, "ms_per_step": cpp_s * 1e3,
               "api": "cals::cp_cals of libcals.so (examples/bench_e2e.cpp): host clock around the call, slowest rank",
               "mean_fit": cpp["mean_fit"], "python": py_e2e}
    else:
        e2e = dict({"unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                    "mean_fit": fit_checksum}, **py_e2e)
    e2e["fraction_of_resident_value"] = e2e["value"] / value

    if rank != 0:
        return None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": done_w,
        "ms_per_step": ev_ms / steps, "higher_is_better": True, "scaling": "strong" if strong else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s, %d forced ALS iterations per model per step%s"
                               % (cfg["name"], als_iters, ", NNLS update" if args.nnls else ""),
                   "total_models": total_models, "models_on_rank0": n_models, "sum_ranks_on_rank0": C,
                   "als_iters_per_step": als_iters,
                   "parallelism": ("ONE model set of %d models sharded over %d GPU(s) by sum of ranks (strong scaling), "
                                   "tensor replicated, no data-path collective" % (total_models, world)) if strong else
                                  ("one full model set per GPU on %d GPU(s) (weak scaling), tensor replicated, no "
                                   "data-path collective" % world),
                   "l2": ("inputs larger than L2: every ALS iteration streams both device copies of the tensor "
                          "(2 x %.0f MB) plus the partial-tile workspace; no explicit flush" % (nX * 8 / 1e6))
                   if 2 * nX * 8 > 126e6 else
                   ("working set (2 x %.0f MB tensor copies) fits the 126 MB L2 -- that is this workload's "
                    "steady state inside cp_cals, not a cache artefact of the timing loop" % (nX * 8 / 1e6))},
        "wall_ms_per_step": wall / steps * 1e3,
        "timing": "CUDA events on the engine's stream around the K steps (barrier + synchronize on both sides), "
                  "max over ranks",
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "e2e": e2e,
    }
    if parity is not None:
        line["parity"] = parity
    if main_line and not args.no_cpu_baseline and world == 1:
        try:
            line["cpu_baseline"] = cpu_baseline(cfg, X, all_models, all_jk)
        except Exception as e:  # the baseline is reported, never allowed to break the bench line
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference",
                                    "sample": "failed: %s" % e}
    return line


def run_sliced(args, cfg_id, rank, world, local_rank, D, steps, warmup, dump_dir=None):
    """BASELINE config 5: ONE tensor sliced over the ranks (strong scaling), all models replicated."""
    import importlib

    import torch
    cfg = CONFIGS[cfg_id]
    sampler = ClockSampler(local_rank).start()
    pkg = load_pkg()
    dmod = importlib.import_module("cp_cals_b200.distributed")
    modes, s_mode, als_iters = cfg["modes"], cfg["sliced"], cfg["als_iters"]
    lo, hi = dmod.shard_slabs(modes[s_mode], world)[rank]
    shape = tuple((hi - lo) if n == s_mode else m for n, m in enumerate(modes))
    # the slab of a seeded uniform(-1,1) tensor: slab r is drawn from its own stream so ranks generate in parallel
    t = torch.empty(int(np.prod(shape)), dtype=torch.float64, pin_memory=True)
    slab = t.numpy().reshape(shape, order="F")
    rng = np.random.default_rng(5000 + rank)
    chunk = 1 << 24
    flat = t.numpy()
    for o in range(0, flat.size, chunk):
        flat[o:o + chunk] = rng.uniform(-1.0, 1.0, size=min(chunk, flat.size - o))
    mrng = np.random.default_rng(77)  # the same models on every rank
    models = []
    for r in cfg["ranks"]:
        fs = []
        for i in modes:
            F = mrng.uniform(-1.0, 1.0, size=(i, r))
            fs.append(np.asfortranarray(F / np.linalg.norm(F, axis=0)))
        models.append(fs)
    C, n_models = sum(cfg["ranks"]), len(models)
    params = pkg.CalsParams(max_iterations=als_iters, buffer_size=C, force_max_iter=True)

    eng = pkg.Engine(local_rank)
    es = torch.cuda.ExternalStream(eng.stream_handle(), device=torch.device("cuda", local_rank))

    def timed(fn, n):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        D.barrier()
        t0 = time.perf_counter()
        ev0.record(es)
        out = [fn() for _ in range(n)]
        ev1.record(es)
        D.barrier()
        return ev0.elapsed_time(ev1), time.perf_counter() - t0, out

    def e2e_step():
        kts = [pkg.Ktensor(list(fs)) for fs in models]
        return dmod.cp_cals_sliced(slab, modes, s_mode, kts, params, engine=eng, device=local_rank), kts

    e2e_step()  # allocations, IPC mapping, upload (untimed)
    sampler.wait_first_sample()
    for _ in range(warmup):
        eng.rerun()
    ev_ms, wall, reps = timed(eng.rerun, steps)
    clocks = sampler.stop()
    if dump_dir and rank == 0:
        dump_outputs(eng, dump_dir)
    ev_ms, wall = D.max(ev_ms), D.max(wall)
    value = n_models * als_iters * steps / (ev_ms * 1e-3)
    launches = sum(r.kernel_launches for r in reps)

    eng.set_timing(1)
    rep = eng.rerun()
    eng.set_timing(0)
    # tensor-sized contractions of the slab: one per mode, or -- slab cut along mode 1 or 2, pair node -- two per iteration
    flops_per_launch = 2.0 * float(np.prod(shape)) * C
    tensor_launches = rep.tensor_flops / flops_per_launch
    mt_ms = D.max(rep.mttkrp_ms - rep.pair_leaf_ms) / tensor_launches
    peak, peak_src = fp64_peak()
    ach = flops_per_launch / (mt_ms * 1e-3) / 1e12
    # NVLink volume of the exchange: every GPU pulls the partials of the other W-1 GPUs (full-size for the modes that
    # are not sliced, the foreign row blocks for the sliced one)
    ld = [(m + 1) // 2 * 2 for m in modes]
    pulled = [8.0 * C * ((modes[n] - (hi - lo)) if n == s_mode else (world - 1) * ld[n]) for n in range(len(modes))]
    xch_ms = D.max(rep.exchange_ms) / rep.mttkrp_launches
    exchange = {"kernel": "exchange_sum_kernel (barrier wait + peer-memory pulls + rank-ordered sum)",
                "ms_per_launch": xch_ms, "nvlink_bytes_pulled_per_gpu_per_launch": float(np.mean(pulled)),
                "achieved_gbs_incl_barrier_wait": float(np.mean(pulled)) / (xch_ms * 1e-3) / 1e9 if xch_ms > 0 else None,
                "peer_copy_peak_gbs": 770.0, "share_of_mttkrp_window": rep.exchange_ms / rep.mttkrp_ms
                if rep.mttkrp_ms > 0 else None} if world > 1 else None
    roofline = {"bound": "tensor", "kernel": "mttkrp_dmma_kernel (+ reduce + NVLink exchange_sum_kernel)" +
                          (" and pair_gemm_kernel" if rep.tree else ""),
                "pair_node": {"contractions_per_als_iteration": tensor_launches / rep.iter,
                              "leaf_ms_per_launch_incl_exchange": D.max(rep.pair_leaf_ms) / (2 * rep.iter),
                              "pair_gemm_ms_per_launch": D.max(rep.pair_gemm_ms) / rep.iter} if rep.tree else None,
                "exchange": exchange,
                "achieved": ach, "peak": peak, "unit": "TFLOP/s per GPU", "frac": ach / peak, "traffic": None,
                "peak_source": peak_src, "ms_per_launch": mt_ms, "flops_per_launch_per_gpu": flops_per_launch,
                "mttkrp_share_of_step": rep.mttkrp_ms / (rep.mttkrp_ms + rep.update_ms)}

    e2e_steps = 2
    e2e_ms, e2e_wall, outs = timed(e2e_step, e2e_steps)
    e2e_t = max(D.max(e2e_ms) * 1e-3, D.max(e2e_wall))
    kts = outs[-1][1]
    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ev_ms / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "%s, %d forced ALS iterations per model per step" % (cfg["name"], als_iters),
                       "models": n_models, "sum_ranks": C, "slab_per_gpu": list(shape),
                       "parallelism": "tensor sliced along mode %d over %d GPU(s), models replicated, one peer-memory "
                                      "exchange per mode" % (s_mode, world),
                       "l2": "inputs larger than L2 (%.1f GB of tensor per GPU)" % (np.prod(shape) * 16 / 1e9)},
            "wall_ms_per_step": wall / steps * 1e3,
            "timing": "CUDA events on the engine's stream around the K steps, max over ranks",
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
            "e2e": {"value": n_models * als_iters * e2e_steps / e2e_t, "unit": UNIT,
                    "h2d_bytes_per_step": int(slab.nbytes + sum(F.nbytes for fs in models for F in fs)),
                    "d2h_bytes_per_step": int(sum(F.nbytes for fs in models for F in fs) + 8 * C),
                    "steps": e2e_steps, "ms_per_step": e2e_t / e2e_steps * 1e3,
                    "api": "cp_cals_sliced of the Python host layer (one process per GPU)",
                    "mean_fit": float(np.mean([k.fit for k in kts]))},
            "cpu_baseline": {"value": None, "unit": UNIT, "cores": 0, "kind": "reference",
                             "sample": "not run: the reference materialises a 10 GB Khatri-Rao workspace for this "
                                       "tensor (SURVEY 8d); config 2 carries the CPU baseline"},
        }
    dmod.release_sliced_engine(eng)
    del t, slab, flat
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=None, choices=sorted(CONFIGS),
                    help="run this configuration only (default: config 2 as the headline, the others as `secondary`)")
    ap.add_argument("--weak", action="store_true", help="N > 1: every rank fits its own full model set (weak scaling) "
                    "instead of sharding ONE model set over the ranks")
    ap.add_argument("--strong", action="store_true", help="accepted for compatibility: strong scaling is the default")
    ap.add_argument("--no-secondary", action="store_true", help="headline configuration only")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--shard-of", type=int, default=0, help="tuning aid on ONE GPU: run only the first shard of an "
                    "N-way split (what each GPU of an N-GPU job gets)")
    ap.add_argument("--no-pair-node", action="store_true", help="measurement aid: one full MTTKRP per mode (3-mode "
                    "tensors otherwise share one contraction between modes 1 and 2, csrc/pairnode.cuh)")
    ap.add_argument("--nnls", action="store_true", help="measurement aid: update_method = NNLS instead of the Cholesky solve")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the fitted models of the headline run's "
                    "last timed step to DIR/<name>.npy (float64) for output-for-output comparison of builds; on N > 1 "
                    "GPUs, rank 0's share of the model set")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    main_cfg = args.config if args.config is not None else 2
    cfg = CONFIGS[main_cfg]

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if cfg.get("sliced") is not None:
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": "config 5 is not run through the CPU reference "
                                  "(10 GB Khatri-Rao workspace); use --config 2"}), flush=True)
            return
        reference_arm(args, cfg, rank)
        return

    steps = args.steps if args.steps is not None else 10
    warmup = max(3, args.warmup if args.warmup is not None else 3)

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = init_nccl(local_rank) if world > 1 else None
    D = Dist(dist)

    def run(cfg_id, st, wu, main_line):
        dump_dir = args.dump_outputs if main_line else None
        if CONFIGS[cfg_id].get("sliced") is not None:
            return run_sliced(args, cfg_id, rank, world, local_rank, D, st, wu, dump_dir)
        return run_sharded(args, cfg_id, rank, world, local_rank, D, st, wu, main_line, dump_dir)

    line = run(main_cfg, steps, warmup, True)
    secondary = []
    if args.config is None and not args.no_secondary and not args.shard_of:
        # the other shapes north_star names, at this GPU count: shorter runs (they only have to be long enough to time)
        for cid in (4, 3, 1, 5):
            st = {4: min(steps, 5), 3: min(steps, 5), 1: min(steps, 10), 5: min(steps, 3)}[cid]
            t0 = time.perf_counter()
            try:
                sec = run(cid, st, 3, False)
            except Exception as e:  # a secondary entry never breaks the headline line
                sec = {"config": {"workload": CONFIGS[cid]["name"]}, "error": "%s: %s" % (type(e).__name__, e)}
                if world > 1:
                    raise  # ranks would fall out of step: let torchrun report it
            if rank == 0 and sec is not None:
                sec["bench_wall_s"] = time.perf_counter() - t0
                secondary.append(sec)
    if rank == 0:
        if secondary:
            line["secondary"] = secondary
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
