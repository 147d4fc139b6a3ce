"""bench.py keeps the driver's contract: one JSON line with the agreed keys, for both arms."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e"}


def _last_json(text):
    lines = [l for l in text.splitlines() if l.startswith("{")]
    assert lines, text[-2000:]
    return json.loads(lines[-1])


def test_reference_arm_line():
    """--impl reference: the unmodified reference (oracle/_ref) on the host cores, bounded sample; runs on CPU."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import caseio
    if not caseio.ref_available():
        pytest.skip("oracle/_ref not built")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = _last_json(out.stdout)
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["metric"] == json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"].split(";")[0]
    assert d["value"] > 0 and d["unit"] == "model-iterations/s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


@pytest.mark.gpu
def test_our_arm_line(tmp_path):
    """The default invocation, shortened: headline config 2 with parity against the unmodified reference, CPU
    baseline, and one `secondary` entry per other BASELINE configuration; --dump-outputs writes the fitted models."""
    dump = tmp_path / "outputs"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3",
                          "--dump-outputs", str(dump)], capture_output=True, text=True, timeout=1500)
    assert out.returncode == 0, out.stderr[-2000:]
    d = _last_json(out.stdout)
    assert BASE_KEYS | {"roofline", "clocks", "gpu_launches"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] >= 3 and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert d["vs_baseline"] is None and d["scaling"] == "strong" and d["config"]["total_models"] == 200
    assert d["clocks"]["samples"] > 0
    r = d["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert 0.5 < r["frac"] < 1.05 and "traffic" in r and (r["traffic"] is None or r["traffic"] > 7e7)
    assert r["traffic"] is not None or "traffic_source" in r  # a stale capture is refused with a reason, not reported
    assert abs(sum(r["share_of_step"].values()) - 1.0) < 0.25 and r["limiter"] in r["share_of_step"]
    e = d["e2e"]
    assert 0 < e["value"] <= d["value"] * 1.02 and e["h2d_bytes_per_step"] > 6e7 and e["d2h_bytes_per_step"] > 1e6
    assert "cals::cp_cals" in e["api"] and e["python"]["value"] > 0
    assert d["gpu_launches"] > 0 and "workload" in d["config"]
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import caseio
    if caseio.ref_available():
        p = d["parity"]
        assert p["ok"] and p["max_rel_err"] <= 1e-9 and p["models"] == 200 and p["iters"] >= 2
        cb = d["cpu_baseline"]
        assert cb["kind"] == "reference" and cb["value"] > 0 and cb["marginal_value"] >= cb["value"] * 0.99
    sec = d["secondary"]
    assert len(sec) == 4 and all("error" not in s for s in sec), [s.get("error") for s in sec]
    for s in sec:
        assert s["value"] > 0 and s["unit"] == "model-iterations/s" and s["clocks"]["samples"] > 0
        assert 0.05 < s["roofline"]["frac"] < 1.05 and s["e2e"]["value"] > 0
    assert any("1000x1000x1000" in s["config"]["workload"] for s in sec)
    import numpy as np
    got = {p.stem: np.load(p) for p in dump.glob("*.npy")}
    C = d["config"]["sum_ranks_on_rank0"]
    shapes = {"factors_mode0": (200, C), "factors_mode1": (200, C), "factors_mode2": (200, C), "lambda": (C,),
              "iters": (200,), "error": (200,), "fit": (200,)}
    assert {k: v.shape for k, v in got.items()} == shapes
    assert all(v.dtype == np.float64 and np.isfinite(v).all() for v in got.values())
    assert sum(v.nbytes for v in got.values()) <= 64 << 20
    assert (got["iters"] == d["config"]["als_iters_per_step"]).all() and (got["fit"] < 1).all()
    # values, model by model in queue order: the dump against the stored outputs of the CPU oracle on the same seeded
    # workload and iteration count (oracle/make_golden.py full)
    from types import SimpleNamespace
    from helpers import RTOL, assert_sampled_models_close, load_sampled
    ranks = [r for r in range(1, 21) for _ in range(10)]  # bench.CONFIGS[2]
    assert sum(ranks) == C
    offs = np.cumsum([0] + ranks)
    models = [SimpleNamespace(factors=[got["factors_mode%d" % n][:, a:b] for n in range(3)], lam=got["lambda"][a:b],
                              iters=got["iters"][i], error=got["error"][i], fit=got["fit"][i])
              for i, (a, b) in enumerate(zip(offs[:-1], offs[1:]))]
    assert_sampled_models_close(models, load_sampled("bench_config2_step"), rtol=RTOL, what="bench dump")


def test_stale_traffic_profile_is_refused(tmp_path, monkeypatch):
    """roofline.traffic comes from an ncu capture; bench.py only uses it while the capture's kernel fingerprint equals
    that of the sources in the tree (VERDICT r1: the number must not silently go stale)."""
    sys.path.insert(0, ROOT)
    import importlib
    bench = importlib.import_module("bench")
    fp = bench.kernel_fingerprint()
    assert len(fp) == 16 and fp == bench.kernel_fingerprint()
    prof = tmp_path / "profiles"
    prof.mkdir()
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))
    monkeypatch.setattr(bench, "kernel_fingerprint", lambda: fp)
    entry = {"kernel": "mttkrp_dmma_kernel<5,4>", "workload": "config2", "dram_bytes_per_launch": 1.0e8}
    (prof / "traffic_r02.json").write_text(json.dumps({"kernel_fingerprint": fp, "kernels": [entry]}))
    assert bench.stored_traffic("mttkrp_dmma_kernel", "config2")[0] == 1.0e8
    (prof / "traffic_r02.json").write_text(json.dumps({"kernel_fingerprint": "0" * 16, "kernels": [entry]}))
    val, why = bench.stored_traffic("mttkrp_dmma_kernel", "config2")
    assert val is None and "stale" in why
