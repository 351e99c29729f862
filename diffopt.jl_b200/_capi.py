"""ctypes binding of libdiffopt_b200.so (include/diffopt_b200.h) -- the same C ABI a Julia
``ccall`` would use.  There is NO fallback: if the library or a CUDA device is missing,
``load()`` / ``Context()`` raise."""
from __future__ import annotations

import ctypes as C
import os
import weakref

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DIFFOPT_B200_LIB") or os.path.join(HERE, "lib", "libdiffopt_b200.so")   # (override: A/B builds)

HOST, DEVICE = 0, 1
QP_SHARED_MATRICES, QP_SHARED_DIRECTION, QP_PACKED_Q, QP_ASYNC, QP_ALLREDUCE = 1, 2, 4, 8, 16
CONE_ZERO, CONE_NONNEG, CONE_SOC, CONE_PSD, CONE_EXP, CONE_DUAL_EXP, CONE_POW, CONE_DUAL_POW = 0, 1, 2, 3, 4, 5, 6, 7

_lib = None

c_dp = C.POINTER(C.c_double)
c_i64p = C.POINTER(C.c_int64)
c_i32p = C.POINTER(C.c_int32)
vp = C.c_void_p

# name -> (restype, argtypes); mirrors include/diffopt_b200.h one to one
SIGNATURES = {
    "diffopt_b200_version": (C.c_int32, []),
    "diffopt_b200_create": (C.c_int32, [C.c_int32, C.POINTER(vp)]),
    "diffopt_b200_destroy": (C.c_int32, [vp]),
    "diffopt_b200_last_error": (C.c_char_p, [vp]),
    "diffopt_b200_launch_count": (C.c_int64, [vp]),
    "diffopt_b200_stream": (vp, [vp]),
    "diffopt_b200_host_alloc": (C.c_int32, [C.POINTER(vp), C.c_int64]),
    "diffopt_b200_host_free": (C.c_int32, [vp]),
    "diffopt_b200_last_kernel_ms": (C.c_double, [vp]),
    "diffopt_b200_qp_batch_solve": (C.c_int32, [vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32] + [vp] * 17 + [C.c_int32]),
    "diffopt_b200_qp_batch_solve_async": (C.c_int32, [vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32] + [vp] * 17),
    "diffopt_b200_synchronize": (C.c_int32, [vp]),
    "diffopt_b200_qp_batch_last_stats": (C.c_int32, [vp, vp]),
    "diffopt_b200_qp_batch_solve_ex": (C.c_int32, [vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32] + [vp] * 17 + [C.c_int32, C.c_int32]),
    "diffopt_b200_qp_batch_solve_coo": (C.c_int32, [vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32] + [vp] * 17 + [C.c_int32, C.c_int32]),
    "diffopt_b200_qp_batch_shared_grads": (C.c_int32, [vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32] + [vp] * 5 + [C.c_int32, C.c_int32]),
    "diffopt_b200_nccl_unique_id": (C.c_int32, [vp]),
    "diffopt_b200_nccl_init": (C.c_int32, [vp, C.c_int32, C.c_int32, vp]),
    "diffopt_b200_nccl_destroy": (C.c_int32, [vp]),
    "diffopt_b200_qp_batch_setup": (C.c_int32, [vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32] + [vp] * 7 + [C.c_int32]),
    "diffopt_b200_qp_batch_reverse": (C.c_int32, [vp, vp, vp, vp, C.c_int32]),
    "diffopt_b200_qp_batch_forward": (C.c_int32, [vp] * 9 + [C.c_int32]),
    "diffopt_b200_qp_batch_factorize": (C.c_int32, [vp, vp, C.c_int32]),
    "diffopt_b200_qp_batch_reverse_multi": (C.c_int32, [vp, C.c_int64, vp, vp, C.c_int32]),
    "diffopt_b200_qp_batch_forward_multi": (C.c_int32, [vp, C.c_int64] + [vp] * 7 + [C.c_int32]),
    "diffopt_b200_qp_batch_param_grads": (C.c_int32, [vp, vp, C.c_int32] + [vp] * 6 + [C.c_int32]),
    "diffopt_b200_kkt_solve_csc": (C.c_int32, [vp, C.c_int64, vp, vp, vp, C.c_int32, C.c_int64, vp, vp, C.c_int32]),
    "diffopt_b200_sparse_setup": (C.c_int32, [vp, C.c_int64, vp, vp, vp, C.c_int32, vp]),
    "diffopt_b200_sparse_solve": (C.c_int32, [vp, C.c_int64, vp, vp, C.c_int32]),
    "diffopt_b200_sparse_stats": (C.c_int32, [vp, vp]),
    "diffopt_b200_sparse_analyze": (C.c_int32, [C.c_int64, vp, vp, vp, C.c_int32, vp]),
    "diffopt_b200_lsqr_csc": (C.c_int32, [vp, C.c_int64, C.c_int64, vp, vp, vp, C.c_int32, vp, C.c_double,
                                          C.c_double, C.c_double, C.c_int64, vp, vp, C.c_int32]),
    "diffopt_b200_conic_setup": (C.c_int32, [vp, C.c_int64, C.c_int64] + [vp] * 8 + [C.c_int64, vp, vp, C.c_int32]),
    "diffopt_b200_conic_setup_ex": (C.c_int32, [vp, C.c_int64, C.c_int64] + [vp] * 8 + [C.c_int64, vp, vp, vp, C.c_int32]),
    "diffopt_b200_conic_get_vp": (C.c_int32, [vp, vp, C.c_int32]),
    "diffopt_b200_conic_dpi_apply": (C.c_int32, [vp, vp, C.c_int32, vp, C.c_int32]),
    "diffopt_b200_conic_M_apply": (C.c_int32, [vp, vp, C.c_int32, vp, C.c_int32]),
    "diffopt_b200_conic_forward": (C.c_int32, [vp, C.c_int64, vp, vp, vp, vp, vp, C.c_double, C.c_double, C.c_double,
                                               C.c_int64, vp, vp, vp, C.c_int32]),
    "diffopt_b200_conic_reverse": (C.c_int32, [vp, vp, C.c_double, C.c_double, C.c_double, C.c_int64, vp, vp, vp, vp,
                                               C.c_int32]),
    "diffopt_b200_conic_batch_begin": (C.c_int32, [vp, C.c_int64, C.c_int32]),
    "diffopt_b200_conic_batch_add": (C.c_int32, [vp, C.c_int64, C.c_int64] + [vp] * 8 + [C.c_int64, vp, vp, C.c_int32]),
    "diffopt_b200_conic_batch_add_ex": (C.c_int32, [vp, C.c_int64, C.c_int64] + [vp] * 8 + [C.c_int64, vp, vp, vp, C.c_int32]),
    "diffopt_b200_conic_batch_reverse": (C.c_int32, [vp, vp, C.c_double, C.c_double, C.c_double, C.c_int64, vp, vp, vp, vp,
                                                     C.c_int32]),
    "diffopt_b200_sparse_setup_inertia": (C.c_int32, [vp, C.c_int64, vp, vp, vp, C.c_int64, C.c_int64, C.c_double, C.c_int32, vp]),
    "diffopt_b200_param_pullback": (C.c_int32, [vp, C.c_int64, vp, vp, vp, C.c_int64, vp, C.c_int64, vp, C.c_int32]),
}


class CooBatch(C.Structure):
    """diffopt_b200_coo_batch: per-instance sparse triplets (0-based offsets ptr, 1-based I, J) of a direction matrix."""
    _fields_ = [("ptr", vp), ("I", vp), ("J", vp), ("V", vp)]


def load():
    """Loads the shared library (raises if it was not built: run ``python __graft_entry__.py``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "diffopt_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class DiffOptB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"diffopt_b200 error {code}: {msg}")
        self.code = code


class SingularException(ArithmeticError):
    """Mirrors ``LinearAlgebra.SingularException(info)`` thrown by the reference's ``LHS \\ RHS``."""

    def __init__(self, info, instance=None):
        super().__init__(f"SingularException({info})" + (f" in instance {instance}" if instance is not None else ""))
        self.info = info
        self.instance = instance


def ptr(a):
    """void* of a numpy array / torch tensor / None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(vp)
    if hasattr(a, "data_ptr"):
        return vp(a.data_ptr())
    raise TypeError(type(a))


class Context:
    """One ctx per GPU (not thread-safe), owns the stream and all device memory."""

    def __init__(self, device=0):
        self.lib = load()
        h = vp()
        rc = self.lib.diffopt_b200_create(int(device), C.byref(h))
        if rc != 0:
            why = {-2: "no usable CUDA device", -4: "device is not sm_100 (B200)", -1: "bad device index"}.get(rc, "?")
            raise DiffOptB200Error(rc, f"diffopt_b200_create failed ({why}); there is no CPU fallback")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.diffopt_b200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc < 0:
            raise DiffOptB200Error(rc, self.lib.diffopt_b200_last_error(self.h).decode())
        return rc

    @property
    def launch_count(self):
        return int(self.lib.diffopt_b200_launch_count(self.h))

    @property
    def last_kernel_ms(self):
        return float(self.lib.diffopt_b200_last_kernel_ms(self.h))

    def qp_last_stats(self):
        """(instances handed to the pivoted-LU fallback, active-set hint, kernel id) of the last qp_batch call."""
        out = np.zeros(3, dtype=np.int64)
        self.check(self.lib.diffopt_b200_qp_batch_last_stats(self.h, ptr(out)))
        return int(out[0]), int(out[1]), int(out[2])

    @property
    def stream(self):
        return self.lib.diffopt_b200_stream(self.h)


def pinned_empty(shape, dtype=np.float64):
    """numpy array backed by cudaHostAlloc'ed (pinned) memory."""
    lib = load()
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = vp()
    rc = lib.diffopt_b200_host_alloc(C.byref(p), max(n, 8))
    if rc != 0:
        raise DiffOptB200Error(rc, "cudaHostAlloc failed")
    buf = (C.c_char * max(n, 8)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    # the ctypes buffer is the base object every view of `arr` keeps alive: free the pinned block when it dies
    weakref.finalize(buf, lib.diffopt_b200_host_free, p.value)
    return arr
