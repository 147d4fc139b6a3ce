"""CPU tests: the C-ABI library builds, loads, exports every symbol include/cals_b200.h declares, and refuses to run
without a GPU (no fallback).  No compute calls are made here."""
import ctypes
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_library_built_and_exports_header_symbols(pkg):
    if not os.path.exists(pkg.LIB_PATH):
        subprocess.run(["make", "-C", os.path.join(ROOT, "cp-cals_b200")], check=True, capture_output=True)
    header = open(os.path.join(ROOT, "include", "cals_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(cals_b200_[a-z0-9_]+)\s*\(", header)))
    assert len(declared) >= 15
    L = ctypes.CDLL(pkg.LIB_PATH)
    for name in declared:
        assert hasattr(L, name), "libcals_b200.so does not export %s" % name
    assert sorted(declared) == sorted(pkg.ABI_SYMBOLS)
    L.cals_b200_version.restype = ctypes.c_char_p
    assert b"sm_100a" in L.cals_b200_version()


def test_library_contains_sm100a_tensor_core_and_tma_code(pkg):
    """SASS evidence that the hot kernel is what DESIGN.md says: DMMA (FP64 tensor core) and UTMALDG (TMA)."""
    cuobjdump = "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump) or not os.path.exists(pkg.LIB_PATH):
        pytest.skip("cuobjdump or library not available")
    sass = subprocess.run([cuobjdump, "-sass", pkg.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    assert "DMMA.8x8x4" in sass
    assert "UTMALDG" in sass
    assert "SYNCS" in sass  # mbarrier


@pytest.mark.skipif(_have_gpu(), reason="only meaningful on a machine without a GPU")
def test_no_cpu_fallback(pkg):
    with pytest.raises(pkg.CalsB200Error) as e:
        pkg.Engine(0)
    assert "no CPU fallback" in str(e.value) or "CUDA" in str(e.value)


def test_streamk_bookkeeping_host(tmp_path):
    nvcc = "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    exe = str(tmp_path / "streamk_test")
    subprocess.run([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
                    os.path.join(ROOT, "tests", "cpp", "streamk_host_test.cu")], check=True, capture_output=True)
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    assert out.stdout.startswith("OK")


def test_python_ktensor_host_logic(pkg):
    import numpy as np
    rng = np.random.default_rng(0)
    kt = pkg.Ktensor([rng.uniform(-1, 1, size=(i, 3)) for i in (5, 4, 6)])
    T0 = None
    kt.normalize()
    for F in kt.factors:
        assert np.allclose(np.linalg.norm(F, axis=0), 1.0)
    T0 = kt.to_tensor()
    kt.denormalize().normalize()
    assert np.allclose(kt.to_tensor(), T0)
    jk = pkg.generate_jk_ktensors(kt)
    assert len(jk) == 5 and all(m.jk_mode == 0 and m.jk_fiber == i for i, m in enumerate(jk))
    p = pkg.CalsParams()
    assert (p.max_iterations, p.tol, p.buffer_size, p.force_max_iter) == (200, 1e-7, 4200, False)
    with pytest.raises(pkg.CalsB200Error):
        pkg._check_params(pkg.CalsParams(line_search=True, line_search_method="error-checking-parallel"))
    pkg._check_params(pkg.CalsParams(line_search=True))
    with pytest.raises(pkg.CalsB200Error):
        pkg._check_params(pkg.CalsParams(update_method="simplex"))
    pkg._check_params(pkg.CalsParams(update_method="nnls"))
