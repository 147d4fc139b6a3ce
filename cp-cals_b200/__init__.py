"""cp-cals_b200: Python host side of the B200-native CP-CALS hot path.

Thin ctypes binding of the C ABI (include/cals_b200.h, built into cp-cals_b200/libcals_b200.so) plus a mirror of
the reference's operator interface for this path -- ``cp_cals`` over a tensor and a list of ``Ktensor`` models with
``CalsParams`` (reference include/cals.h:138-198) and ``jk_cp_cals`` (reference src/cals.cpp:397-446).

There is NO CPU fallback here: if the CUDA library is missing or no B200 is visible every call raises.
(The directory name contains a hyphen; import it with ``importlib`` as ``cp_cals_b200`` -- see ``load_package`` in
__graft_entry__.py.)
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CALS_B200_LIB", os.path.join(HERE, "libcals_b200.so"))  # env override: debug builds only

FORCE_MAX_ITER = 1
ALWAYS_EVICT_FIRST = 2
NNLS = 4
MTTKRP_DMMA = 0
MTTKRP_NAIVE = 1

# every symbol include/cals_b200.h declares
ABI_SYMBOLS = [
    "cals_b200_create", "cals_b200_destroy", "cals_b200_last_error", "cals_b200_set_tensor",
    "cals_b200_set_tensor_dev", "cals_b200_configure", "cals_b200_set_timing", "cals_b200_set_mttkrp_variant",
    "cals_b200_clear_models", "cals_b200_enqueue_model", "cals_b200_run", "cals_b200_rerun",
    "cals_b200_fetch_model", "cals_b200_fetch_all", "cals_b200_tensor_norm", "cals_b200_jk_norms",
    "cals_b200_mttkrp", "cals_b200_device_info", "cals_b200_version", "cals_b200_fetch_iteration_cols",
    "cals_b200_host_alloc", "cals_b200_host_free", "cals_b200_stream",
    "cals_b200_comm_alloc", "cals_b200_comm_local_block", "cals_b200_comm_connect", "cals_b200_set_tensor_slab",
    "cals_b200_set_tensor_norm", "cals_b200_comm_disconnect", "cals_b200_set_model_active_set",
    "cals_b200_fetch_model_active_set", "cals_b200_set_line_search", "cals_b200_line_search_counts",
    "cals_b200_enqueue_models", "cals_b200_set_pair_node", "cals_b200_khatri_rao", "cals_b200_core_consistency",
]


class CalsB200Error(RuntimeError):
    pass


class Report(C.Structure):
    """cals_b200_report (include/cals_b200.h) == the CalsReport fields the path fills (reference include/cals.h:27-63)."""

    _fields_ = [("iter", C.c_uint64), ("n_ktensors", C.c_uint64), ("ktensor_comp_sum", C.c_uint64),
                ("x_norm", C.c_double), ("total_time", C.c_double), ("device_ms", C.c_double),
                ("mttkrp_ms", C.c_double), ("update_ms", C.c_double), ("mttkrp_launches", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("mttkrp_flops", C.c_double), ("exchange_ms", C.c_double),
                ("pair_gemm_ms", C.c_double), ("pair_leaf_ms", C.c_double), ("tensor_flops", C.c_double),
                ("tree", C.c_int32), ("fused_leaf_blocks", C.c_int32), ("sweep_period", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class ModelStats(C.Structure):
    _fields_ = [("iters", C.c_uint64), ("error", C.c_double), ("fit", C.c_double), ("old_fit", C.c_double),
                ("chol_info", C.c_int32)]


_lib = None


def lib():
    """Load libcals_b200.so (fails loudly when it has not been built: there is no fallback path)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CalsB200Error("%s not found: build it with `make -C cp-cals_b200` (or __graft_entry__.build())" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i, u64, dbl = C.c_void_p, C.c_int, C.c_uint64, C.c_double
    L.cals_b200_create.argtypes = [C.POINTER(vp), i]
    L.cals_b200_destroy.argtypes = [vp]
    L.cals_b200_last_error.argtypes = [vp]
    L.cals_b200_last_error.restype = C.c_char_p
    L.cals_b200_set_tensor.argtypes = [vp, i, C.POINTER(u64), vp]
    L.cals_b200_set_tensor_dev.argtypes = [vp, i, C.POINTER(u64), vp]
    L.cals_b200_configure.argtypes = [vp, u64, u64, dbl, C.c_uint]
    L.cals_b200_set_timing.argtypes = [vp, i]
    L.cals_b200_set_mttkrp_variant.argtypes = [vp, i]
    L.cals_b200_set_pair_node.argtypes = [vp, i]
    L.cals_b200_clear_models.argtypes = [vp]
    L.cals_b200_enqueue_model.argtypes = [vp, u64, C.POINTER(vp), i, C.c_int64, C.POINTER(i)]
    L.cals_b200_run.argtypes = [vp, C.POINTER(Report)]
    L.cals_b200_rerun.argtypes = [vp, C.POINTER(Report)]
    L.cals_b200_fetch_model.argtypes = [vp, i, C.POINTER(vp), vp, C.POINTER(ModelStats)]
    L.cals_b200_fetch_all.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(ModelStats)]
    L.cals_b200_tensor_norm.argtypes = [vp, C.POINTER(dbl)]
    L.cals_b200_jk_norms.argtypes = [vp, vp]
    L.cals_b200_mttkrp.argtypes = [vp, i, u64, C.POINTER(vp), vp, i, i, C.POINTER(dbl)]
    L.cals_b200_device_info.argtypes = [vp, C.POINTER(i), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    L.cals_b200_version.restype = C.c_char_p
    L.cals_b200_fetch_iteration_cols.argtypes = [vp, C.POINTER(C.c_uint32), u64, C.POINTER(u64)]
    L.cals_b200_host_alloc.argtypes = [C.c_size_t]
    L.cals_b200_host_alloc.restype = vp
    L.cals_b200_host_free.argtypes = [vp]
    L.cals_b200_stream.argtypes = [vp, C.POINTER(vp)]
    L.cals_b200_comm_alloc.argtypes = [vp, i, i, u64, vp]
    L.cals_b200_comm_local_block.argtypes = [vp, C.POINTER(vp)]
    L.cals_b200_comm_connect.argtypes = [vp, vp, C.POINTER(vp), C.POINTER(i)]
    L.cals_b200_set_tensor_slab.argtypes = [vp, i, C.POINTER(u64), i, C.POINTER(u64), vp]
    L.cals_b200_set_tensor_norm.argtypes = [vp, dbl]
    L.cals_b200_comm_disconnect.argtypes = [vp]
    L.cals_b200_enqueue_models.argtypes = [vp, u64, C.POINTER(u64), C.POINTER(vp), C.POINTER(i), C.POINTER(C.c_int64)]
    L.cals_b200_set_line_search.argtypes = [vp, i, i, i, dbl]
    L.cals_b200_khatri_rao.argtypes = [vp, vp, u64, vp, u64, u64, vp]
    L.cals_b200_line_search_counts.argtypes = [vp, C.POINTER(u64), C.POINTER(u64)]
    L.cals_b200_set_model_active_set.argtypes = [vp, i, C.POINTER(vp)]
    L.cals_b200_fetch_model_active_set.argtypes = [vp, i, C.POINTER(vp)]
    L.cals_b200_core_consistency.argtypes = [vp, vp, vp]
    _lib = L
    return L


# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class Ktensor:
    """One CP model (reference include/ktensor.h:24-341): factors[n] is (I_n, R) float64, lam is (R,)."""

    factors: List[np.ndarray]
    lam: Optional[np.ndarray] = None
    jk_mode: int = -1
    jk_fiber: int = 0
    iters: int = 0
    error: float = 0.0
    fit: float = 0.0
    old_fit: float = 0.0
    chol_info: int = 0
    active_set: Optional[List[np.ndarray]] = None  # NNLS: per mode (I_n, R) bool, None = all constraints active

    @property
    def rank(self) -> int:
        return int(self.factors[0].shape[1])

    @property
    def fit_diff(self) -> float:  # Ktensor::get_fit_diff, include/ktensor.h:189
        return abs(self.old_fit - self.fit)

    def to_jk(self, mode: int, fiber: int) -> "Ktensor":  # include/ktensor.h:276-282
        self.jk_mode, self.jk_fiber = mode, fiber
        return self

    def copy(self) -> "Ktensor":
        return Ktensor([np.array(F, order="F", copy=True) for F in self.factors],
                       None if self.lam is None else self.lam.copy(), self.jk_mode, self.jk_fiber, self.iters,
                       self.error, self.fit, self.old_fit, self.chol_info)

    def normalize(self) -> "Ktensor":  # Ktensor::normalize(), src/ktensor.cpp:85-99
        lam = np.ones(self.rank)
        for k, F in enumerate(self.factors):
            nrm = np.linalg.norm(F, axis=0)
            self.factors[k] = np.asfortranarray(F * (1.0 / nrm))
            lam = lam * nrm
        self.lam = lam
        return self

    def denormalize(self) -> "Ktensor":  # Ktensor::denormalize, src/ktensor.cpp:101-107
        self.factors[0] = np.asfortranarray(self.factors[0] * self.lam)
        return self

    def set_jk_fiber(self, value: float) -> None:  # include/ktensor.h:316-325
        if self.jk_mode >= 0:
            if np.isnan(value):
                self.factors[self.jk_mode][self.jk_fiber, :] = np.nan
            else:
                self.factors[self.jk_mode][self.jk_fiber, :] *= value

    def to_tensor(self) -> np.ndarray:  # Ktensor::to_tensor, src/ktensor.cpp:51-64
        N = len(self.factors)
        letters = "abcdefgh"[:N]
        expr = ",".join(l + "r" for l in letters) + ",r->" + letters
        return np.einsum(expr, *self.factors, self.lam, optimize=True)


@dataclass
class CalsParams:
    """reference include/cals.h:138-159 (same names, same defaults)."""

    update_method: str = "unconstrained"
    mttkrp_method: str = "auto"  # "mttkrp": one contraction per mode; anything else: shared where possible (pair node)
    max_iterations: int = 200
    tol: float = 1e-7
    cuda: bool = True
    buffer_size: int = 4200
    line_search: bool = False
    line_search_interval: int = 5
    line_search_step: float = 0.0
    line_search_method: str = "no-error-checking"  # | "error-checking-serial" (include/utils/line_search.h:10-11)
    force_max_iter: bool = False
    always_evict_first: bool = False


@dataclass
class CalsReport:
    """The part of reference include/cals.h:27-63 this path fills."""

    n_modes: int = 0
    modes: Sequence[int] = ()
    X_norm: float = 0.0
    iter: int = 0
    max_iter: int = 0
    buffer_size: int = 0
    n_ktensors: int = 0
    ktensor_comp_sum: int = 0
    tol: float = 0.0
    total_time: float = 0.0
    device_ms: float = 0.0
    mttkrp_ms: float = 0.0
    update_ms: float = 0.0
    mttkrp_launches: int = 0
    kernel_launches: int = 0
    ls_performed: int = 0
    ls_failed: int = 0
    pair_node: bool = False  # modes 1 and 2 took their MTTKRP from the shared contraction (csrc/pairnode.cuh)
    tensor_flops: float = 0.0  # flop of the tensor-sized contractions that actually ran
    sweep_period: int = 1  # 2: the multi-sweep dimension tree carried a contraction from one iteration to the next


class Engine:
    """RAII wrapper of one cals_b200_ctx (one per caller thread / per GPU)."""

    def __init__(self, device: int = 0):
        self._L = lib()
        self._ctx = C.c_void_p()
        if self._L.cals_b200_create(C.byref(self._ctx), device) != 0:
            raise CalsB200Error(self._L.cals_b200_last_error(None).decode())
        self.modes = None
        self._keep = []

    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx:
            self._L.cals_b200_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        if rc != 0:
            raise CalsB200Error(self._L.cals_b200_last_error(self._ctx).decode())

    # -- tensor ------------------------------------------------------------------------------------------------------
    def set_tensor(self, X: np.ndarray):
        Xf = np.asfortranarray(X, dtype=np.float64)
        modes = (C.c_uint64 * Xf.ndim)(*Xf.shape)
        self._ck(self._L.cals_b200_set_tensor(self._ctx, Xf.ndim, modes, Xf.ctypes.data))
        self._keep_X = Xf  # the upload is asynchronous: keep the source alive until the next synchronising call
        self.modes = tuple(Xf.shape)

    def set_tensor_dev(self, dev_ptr: int, modes: Sequence[int]):
        m = (C.c_uint64 * len(modes))(*modes)
        self._ck(self._L.cals_b200_set_tensor_dev(self._ctx, len(modes), m, C.c_void_p(dev_ptr)))
        self.modes = tuple(modes)

    # -- tensor sliced over several GPUs (BASELINE config 5) ---------------------------------------------------------
    def comm_alloc(self, rank: int, world: int, capacity_doubles: int) -> bytes:
        """Allocate the exchange block; returns its 64-byte CUDA IPC handle."""
        h = C.create_string_buffer(64)
        self._ck(self._L.cals_b200_comm_alloc(self._ctx, rank, world, capacity_doubles, h))
        self.comm_rank, self.comm_world = rank, world
        return h.raw

    def comm_disconnect(self):
        self._ck(self._L.cals_b200_comm_disconnect(self._ctx))
        self._comm = None

    def comm_local_block(self) -> int:
        out = C.c_void_p()
        self._ck(self._L.cals_b200_comm_local_block(self._ctx, C.byref(out)))
        return int(out.value)

    def comm_connect_ipc(self, handles: Sequence[bytes]):
        blob = b"".join(handles)
        assert len(blob) == 64 * self.comm_world
        self._ck(self._L.cals_b200_comm_connect(self._ctx, blob, None, None))

    def comm_connect_ptr(self, blocks: Sequence[int], devices: Sequence[int]):
        bl = (C.c_void_p * len(blocks))(*blocks)
        dv = (C.c_int * len(devices))(*devices)
        self._ck(self._L.cals_b200_comm_connect(self._ctx, None, bl, dv))

    def set_tensor_slab(self, modes: Sequence[int], slice_mode: int, cuts: Sequence[int], slab: np.ndarray):
        """slab: this rank's part X[..., cuts[rank]:cuts[rank+1], ...] along slice_mode (dense)."""
        Sf = np.asfortranarray(slab, dtype=np.float64)
        want = tuple((cuts[self.comm_rank + 1] - cuts[self.comm_rank]) if n == slice_mode else m
                     for n, m in enumerate(modes))
        if tuple(Sf.shape) != want:
            raise ValueError("slab shape %s does not match %s" % (Sf.shape, want))
        m = (C.c_uint64 * len(modes))(*modes)
        cu = (C.c_uint64 * len(cuts))(*cuts)
        self._ck(self._L.cals_b200_set_tensor_slab(self._ctx, len(modes), m, slice_mode, cu, Sf.ctypes.data))
        self._keep_X = Sf
        self.modes = tuple(modes)

    def set_tensor_norm(self, norm: float):
        self._ck(self._L.cals_b200_set_tensor_norm(self._ctx, norm))

    def tensor_norm(self) -> float:
        out = C.c_double()
        self._ck(self._L.cals_b200_tensor_norm(self._ctx, C.byref(out)))
        return out.value

    def jk_norms(self) -> np.ndarray:
        out = np.zeros(self.modes[0])
        self._ck(self._L.cals_b200_jk_norms(self._ctx, out.ctypes.data))
        return out

    # -- parameters ----------------------------------------------------------------------------------------------------
    def configure(self, buffer_cols: int, max_iterations: int, tol: float, force_max_iter=False,
                  always_evict_first=False, nnls=False):
        flags = ((FORCE_MAX_ITER if force_max_iter else 0) | (ALWAYS_EVICT_FIRST if always_evict_first else 0) |
                 (NNLS if nnls else 0))
        self._ck(self._L.cals_b200_configure(self._ctx, buffer_cols, max_iterations, tol, flags))

    def set_line_search(self, enabled: bool, method: int = 0, interval: int = 5, step: float = 0.0):
        """method 0 = no error checking, 1 = error checking (serial) -- reference include/utils/line_search.h:8."""
        self._ck(self._L.cals_b200_set_line_search(self._ctx, 1 if enabled else 0, method, interval, step))

    def line_search_counts(self):
        a, b = C.c_uint64(), C.c_uint64()
        self._ck(self._L.cals_b200_line_search_counts(self._ctx, C.byref(a), C.byref(b)))
        return a.value, b.value

    def set_timing(self, level: int):
        self._ck(self._L.cals_b200_set_timing(self._ctx, level))

    def set_mttkrp_variant(self, variant: int):
        self._ck(self._L.cals_b200_set_mttkrp_variant(self._ctx, variant))

    def set_pair_node(self, enabled: bool):
        self._ck(self._L.cals_b200_set_pair_node(self._ctx, int(bool(enabled))))

    # -- queue -----------------------------------------------------------------------------------------------------------
    def clear_models(self):
        self._ck(self._L.cals_b200_clear_models(self._ctx))
        self._ranks = []

    def enqueue(self, factors: Sequence[np.ndarray], jk_mode: int = -1, jk_fiber: int = 0) -> int:
        fs = [np.asfortranarray(F, dtype=np.float64) for F in factors]
        rank = fs[0].shape[1]
        for F, I in zip(fs, self.modes):
            if F.shape != (I, rank):
                raise ValueError("factor shape %s does not match (%d, %d)" % (F.shape, I, rank))
        ptrs = (C.c_void_p * len(fs))(*[F.ctypes.data for F in fs])
        mid = C.c_int()
        self._ck(self._L.cals_b200_enqueue_model(self._ctx, rank, ptrs, jk_mode, jk_fiber, C.byref(mid)))
        if not hasattr(self, "_ranks"):
            self._ranks = []
        self._ranks.append(rank)
        return mid.value

    def enqueue_many(self, models: Sequence[Sequence[np.ndarray]], jk: Optional[Sequence[tuple]] = None):
        """Queue a list of models with one call through the C ABI.  models[m][n] is (I_n, R_m); jk[m] = (mode, fiber)
        or (-1, 0).  The arrays must be float64; Fortran-ordered ones are passed as they are (no copy)."""
        N = len(self.modes)
        keep, ptrs, ranks = [], [], []
        for fs in models:
            if len(fs) != N:
                raise ValueError("a model has %d factors, the tensor has %d modes" % (len(fs), N))
            R = fs[0].shape[1]
            ranks.append(R)
            for F, I in zip(fs, self.modes):
                if F.shape != (I, R):
                    raise ValueError("factor shape %s does not match (%d, %d)" % (F.shape, I, R))
                if F.dtype != np.float64 or not F.flags.f_contiguous:
                    F = np.asfortranarray(F, dtype=np.float64)
                    keep.append(F)
                ptrs.append(F.ctypes.data)
        M = len(ranks)
        a_ranks = (C.c_uint64 * M)(*ranks)
        a_ptrs = (C.c_void_p * (M * N))(*ptrs)
        a_jm = a_jf = None
        if jk is not None and any(j[0] >= 0 for j in jk):
            a_jm = (C.c_int * M)(*[j[0] for j in jk])
            a_jf = (C.c_int64 * M)(*[j[1] for j in jk])
        self._ck(self._L.cals_b200_enqueue_models(self._ctx, M, a_ranks, a_ptrs, a_jm, a_jf))
        if not hasattr(self, "_ranks"):
            self._ranks = []
        self._ranks.extend(ranks)

    # -- run ---------------------------------------------------------------------------------------------------------------
    def run(self) -> Report:
        rep = Report()
        self._ck(self._L.cals_b200_run(self._ctx, C.byref(rep)))
        return rep

    def rerun(self) -> Report:
        rep = Report()
        self._ck(self._L.cals_b200_rerun(self._ctx, C.byref(rep)))
        return rep

    def fetch(self, model_id: int):
        rank = self._ranks[model_id]
        fs = [np.zeros((I, rank), order="F") for I in self.modes]
        lam = np.zeros(rank)
        ptrs = (C.c_void_p * len(fs))(*[F.ctypes.data for F in fs])
        st = ModelStats()
        self._ck(self._L.cals_b200_fetch_model(self._ctx, model_id, ptrs, lam.ctypes.data, C.byref(st)))
        return fs, lam, st

    def set_active_set(self, model_id: int, active: Sequence[np.ndarray]):
        """active[n]: (I_n, R) bool/uint8, True = entry constrained to zero (Ktensor::active_set of the reference)."""
        arrs = [np.ascontiguousarray(a, dtype=np.uint8) for a in active]
        ptrs = (C.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
        self._ck(self._L.cals_b200_set_model_active_set(self._ctx, model_id, ptrs))

    def fetch_active_set(self, model_id: int):
        R = self._ranks[model_id]
        arrs = [np.empty((I, R), dtype=np.uint8) for I in self.modes]
        ptrs = (C.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
        self._ck(self._L.cals_b200_fetch_model_active_set(self._ctx, model_id, ptrs))
        return [a.astype(bool) for a in arrs]

    def fetch_all(self):
        """All models of the last run with ONE call through the C ABI: [(factors, lam, stats), ...] in queue order."""
        M, N = len(self._ranks), len(self.modes)
        # one allocation per mode (and one for lambda) holding all models side by side; every model gets column views
        total = sum(self._ranks)
        big = [np.empty((I, total), order="F") for I in self.modes]
        lam_all = np.empty(total)
        base = [b.ctypes.data for b in big]
        lbase = lam_all.ctypes.data
        fptr = (C.c_void_p * (M * N))()
        lptr = (C.c_void_p * M)()
        fs, lams, col = [], [], 0
        for m, r in enumerate(self._ranks):
            fs.append([b[:, col:col + r] for b in big])
            lams.append(lam_all[col:col + r])
            for n, I in enumerate(self.modes):
                fptr[m * N + n] = base[n] + 8 * I * col
            lptr[m] = lbase + 8 * col
            col += r
        stats = (ModelStats * M)()
        self._ck(self._L.cals_b200_fetch_all(self._ctx, fptr, lptr, stats))
        return [(fs[m], lams[m], stats[m]) for m in range(M)]

    def core_consistency(self):
        """Core consistency (CORCONDIA) of every queued model: (cc, status), one entry per model in queue order.  After
        run / rerun it scores the fitted models, before any run the enqueued factors with lambda = 1.  status 0 =
        computed, 1 = rank above the limit (96 for 3 modes, 64 for 4), 2 = a Gram matrix A_n^T A_n is not positive
        definite; cc is NaN unless status is 0."""
        M = len(getattr(self, "_ranks", []))
        cc = np.empty(M)
        status = np.empty(M, dtype=np.int32)
        self._ck(self._L.cals_b200_core_consistency(self._ctx, cc.ctypes.data, status.ctypes.data))
        return cc, status

    # -- hooks ---------------------------------------------------------------------------------------------------------------
    def mttkrp(self, factors: Sequence[np.ndarray], mode: int, variant: int = MTTKRP_DMMA, repeats: int = 1):
        """G = X_(mode) * KRP(factors except mode) over the concatenated columns.  Returns (G, ms_per_launch)."""
        fs = [None if k == mode else np.asfortranarray(F, dtype=np.float64) for k, F in enumerate(factors)]
        cols = fs[(mode + 1) % len(fs)].shape[1]
        ptrs = (C.c_void_p * len(fs))(*[None if F is None else F.ctypes.data for F in fs])
        G = np.zeros((self.modes[mode], cols), order="F")
        ms = C.c_double()
        self._ck(self._L.cals_b200_mttkrp(self._ctx, mode, cols, ptrs, G.ctypes.data, variant, repeats, C.byref(ms)))
        return G, ms.value

    def khatri_rao(self, A: np.ndarray, B: np.ndarray) -> np.ndarray:
        """mttkrp::khatri_rao (reference src/utils/mttkrp.cpp:78-103): K[ib + IB*ia, c] = A[ia, c] * B[ib, c]."""
        Af, Bf = np.asfortranarray(A, dtype=np.float64), np.asfortranarray(B, dtype=np.float64)
        if Af.ndim != 2 or Bf.ndim != 2 or Af.shape[1] != Bf.shape[1]:
            raise ValueError("khatri_rao needs two matrices with the same number of columns")
        K = np.empty((Af.shape[0] * Bf.shape[0], Af.shape[1]), order="F")
        self._ck(self._L.cals_b200_khatri_rao(self._ctx, Af.ctypes.data, Af.shape[0], Bf.ctypes.data, Bf.shape[0],
                                              Af.shape[1], K.ctypes.data))
        return K

    def iteration_cols(self) -> np.ndarray:
        """CalsReport::cols of the last run: active multi-factor columns per global iteration."""
        n = C.c_uint64()
        self._ck(self._L.cals_b200_fetch_iteration_cols(self._ctx, None, 0, C.byref(n)))
        out = np.zeros(n.value, dtype=np.uint32)
        if n.value:
            self._ck(self._L.cals_b200_fetch_iteration_cols(self._ctx, out.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                            n.value, C.byref(n)))
        return out

    def stream_handle(self) -> int:
        """cudaStream_t of this context as an integer (wrap with torch.cuda.ExternalStream to record events on it)."""
        out = C.c_void_p()
        self._ck(self._L.cals_b200_stream(self._ctx, C.byref(out)))
        return int(out.value or 0)

    def device_info(self):
        sm, fr, tot = C.c_int(), C.c_size_t(), C.c_size_t()
        self._ck(self._L.cals_b200_device_info(self._ctx, C.byref(sm), C.byref(fr), C.byref(tot)))
        return {"sm_count": sm.value, "free_bytes": fr.value, "total_bytes": tot.value}


# ---------------------------------------------------------------------------------------------------------------------
LS_METHODS = {"no-error-checking": 0, "error-checking-serial": 1}


def _check_params(params: CalsParams):
    if params.update_method not in ("unconstrained", "nnls"):
        raise CalsB200Error("unknown update_method %r (reference include/utils/update.h:8: unconstrained | nnls)"
                            % (params.update_method,))
    if params.line_search and params.line_search_method not in LS_METHODS:
        raise CalsB200Error("line search method %r is not available (%s)" % (params.line_search_method,
                                                                             " | ".join(LS_METHODS)))


def cp_cals(X: np.ndarray, ktensors: Sequence[Ktensor], params: CalsParams, *, engine: Optional[Engine] = None,
            device: int = 0, timing: int = 0, mttkrp_variant: int = MTTKRP_DMMA) -> CalsReport:
    """cals::cp_cals (reference src/cals.cpp:19-395): fit every model of `ktensors` (consumed FIFO) to X concurrently;
    each Ktensor is overwritten in place with its fitted factors, lambda, error, fit and iteration count."""
    _check_params(params)
    own = engine is None
    eng = engine or Engine(device)
    try:
        if own or eng.modes is None or X is not None:
            eng.set_tensor(X)
        nnls = params.update_method == "nnls"
        eng.configure(params.buffer_size, params.max_iterations, params.tol, params.force_max_iter,
                      params.always_evict_first, nnls)
        eng.set_line_search(params.line_search, LS_METHODS.get(params.line_search_method, 0),
                            params.line_search_interval, params.line_search_step)
        eng.set_timing(timing)
        eng.set_mttkrp_variant(mttkrp_variant)
        eng.set_pair_node(str(params.mttkrp_method).lower() != "mttkrp")
        eng.clear_models()
        eng.enqueue_many([kt.factors for kt in ktensors], [(kt.jk_mode, kt.jk_fiber) for kt in ktensors])
        if nnls:  # active sets persist in the Ktensor across calls (reference include/ktensor.h:36)
            for i, kt in enumerate(ktensors):
                if kt.active_set is not None:
                    eng.set_active_set(i, kt.active_set)
        rep = eng.run()
        for i, (kt, (fs, lam, st)) in enumerate(zip(ktensors, eng.fetch_all())):
            kt.factors, kt.lam = fs, lam
            kt.iters, kt.error, kt.fit, kt.old_fit, kt.chol_info = st.iters, st.error, st.fit, st.old_fit, st.chol_info
            if nnls:
                kt.active_set = eng.fetch_active_set(i)
        lsp, lsf = eng.line_search_counts()
        return CalsReport(n_modes=X.ndim, modes=tuple(X.shape), X_norm=rep.x_norm, iter=rep.iter,
                          max_iter=params.max_iterations, buffer_size=params.buffer_size, n_ktensors=rep.n_ktensors,
                          ktensor_comp_sum=rep.ktensor_comp_sum, tol=params.tol, total_time=rep.total_time,
                          device_ms=rep.device_ms, mttkrp_ms=rep.mttkrp_ms, update_ms=rep.update_ms,
                          mttkrp_launches=rep.mttkrp_launches, kernel_launches=rep.kernel_launches,
                          ls_performed=lsp, ls_failed=lsf, pair_node=bool(rep.tree), tensor_flops=rep.tensor_flops,
                          sweep_period=rep.sweep_period)
    finally:
        if own:
            eng.close()


def core_consistency(X: Optional[np.ndarray], ktensors: Sequence[Ktensor], engine: Optional[Engine] = None,
                     device: int = 0) -> np.ndarray:
    """Core consistency (Bro & Kiers 2003) of every Ktensor against X, on the device: lambda (when set) is folded into
    mode 0, jackknife flags are kept (the model leaves out its row of mode 0).  Returns one value per model, NaN for a
    model whose rank is above the limit or whose factors are rank-deficient (Engine.core_consistency has the status)."""
    own = engine is None
    eng = engine or Engine(device)
    try:
        if own or eng.modes is None or X is not None:
            eng.set_tensor(X)
        eng.clear_models()
        models = []
        for kt in ktensors:
            fs = list(kt.factors)
            if kt.lam is not None:
                fs[0] = np.asfortranarray(fs[0] * np.asarray(kt.lam)[None, :])
            models.append(fs)
        eng.enqueue_many(models, [(kt.jk_mode, kt.jk_fiber) for kt in ktensors])
        return eng.core_consistency()[0]
    finally:
        if own:
            eng.close()


def generate_jk_ktensors(reference: Ktensor) -> List[Ktensor]:
    """utils::generate_jk_ktensors (reference src/utils/utils.cpp:40-51): one copy per mode-0 sample, flagged."""
    I0 = reference.factors[0].shape[0]
    if I0 <= 1:
        raise CalsB200Error("Can't do Jack-knife with just one sample.")
    return [reference.copy().to_jk(0, i) for i in range(I0)]


def jk_cp_cals(X: np.ndarray, ktensors: Sequence[Ktensor], params: CalsParams, **kw):
    """cals::jk_cp_cals (reference src/cals.cpp:397-446) up to, and excluding, the LSAP column matching
    (jk_permutation_adjustment, src/utils/utils.cpp:53-101: host post-processing, SURVEY section 8f-1).
    Returns (report, results) with results[b][i] the leave-sample-i-out model of base model b."""
    bases = [kt.copy().denormalize().normalize() for kt in ktensors]
    jk_input = [generate_jk_ktensors(b) for b in bases]
    flat = [m for group in jk_input for m in group]
    rep = cp_cals(X, flat, params, **kw)
    for m in flat:
        m.set_jk_fiber(0.0)
        m.denormalize()
        m.normalize()
        m.set_jk_fiber(float("nan"))
    return rep, jk_input
