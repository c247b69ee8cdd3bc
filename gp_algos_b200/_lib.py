"""ctypes binding of libgpk.so (include/gpk.h).  Fails loudly when the library or a GPU is missing."""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_dp = C.POINTER(C.c_double)
_i64 = C.c_int64

GPK_OK, GPK_EINVAL, GPK_ENOTSYM, GPK_ENOTPD, GPK_ECUDA, GPK_ENOMEM = 0, -1, -2, -3, -4, -5


class GpkError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"libgpk status {status}: {msg}")
        self.status = status


class IllegalArgumentError(GpkError, ValueError):
    """java.lang.IllegalArgumentException (`require` at GpPredictor.scala:108, MatrixUtils.scala:125)."""


class MatrixNotSymmetricError(GpkError):
    """breeze.linalg.MatrixNotSymmetricException."""


class NotPositiveDefiniteError(GpkError):
    """breeze.linalg.NotConvergedException raised by `cholesky`; .minor = failing leading minor (1-based)."""

    def __init__(self, status, msg, minor):
        super().__init__(status, msg)
        self.minor = minor


def lib_path() -> str:
    return os.path.join(_HERE, "libgpk.so")


_lib = None
_lock = threading.Lock()


def load():
    """Load libgpk.so (built in-tree by __graft_entry__.build() / csrc/Makefile)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = lib_path()
        if not os.path.exists(path):
            raise GpkError(GPK_ECUDA, f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                                      f"(there is no CPU fallback)")
        lib = C.CDLL(path)
        lib.gpk_version.restype = C.c_char_p
        lib.gpk_last_error.restype = C.c_char_p
        lib.gpk_last_error.argtypes = [C.c_void_p]
        lib.gpk_last_info.argtypes = [C.c_void_p]
        lib.gpk_launch_count.restype = C.c_int64
        lib.gpk_launch_count.argtypes = [C.c_void_p]
        lib.gpk_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_void_p]
        lib.gpk_destroy.argtypes = [C.c_void_p]
        lib.gpk_synchronize.argtypes = [C.c_void_p]
        lib.gpk_set_graph_mode.argtypes = [C.c_void_p, C.c_int]
        lib.gpk_set_kernel_family.argtypes = [C.c_void_p, C.c_int]
        lib.gpk_get_kernel_family.argtypes = [C.c_void_p]
        lib.gpk_theta_length.argtypes = [C.c_void_p, C.c_int]
        vp, ci, cd = C.c_void_p, C.c_int, C.c_double
        lib.gpk_cov_se_ard.argtypes = [vp, vp, ci, ci, _i64, vp, vp, _i64]
        lib.gpk_cov_se_ard_dev.argtypes = [vp, vp, ci, ci, _i64, vp, vp, _i64]
        lib.gpk_cov_cross_se_ard.argtypes = [vp, vp, ci, _i64, vp, ci, _i64, ci, vp, vp, _i64]
        lib.gpk_cov_cross_se_ard_dev.argtypes = [vp, vp, ci, _i64, vp, ci, _i64, ci, vp, vp, _i64]
        lib.gpk_cov_deriv_se_ard.argtypes = [vp, ci, vp, ci, ci, _i64, vp, vp, _i64]
        lib.gpk_potrf_lower.argtypes = [vp, vp, ci, _i64, vp, _i64, ci]
        lib.gpk_potrf_lower_dev.argtypes = [vp, vp, ci, _i64, vp]
        lib.gpk_trsm.argtypes = [vp, ci, ci, vp, ci, _i64, vp, ci, _i64, vp, _i64]
        lib.gpk_trtri.argtypes = [vp, ci, vp, ci, _i64, vp, _i64]
        lib.gpk_syrk_lower_dev.argtypes = [vp, vp, _i64, vp, _i64, ci, ci]
        lib.gpk_gp_fit.argtypes = [vp, vp, ci, ci, _i64, vp, vp, ci, cd, vp, _i64, vp, vp]
        lib.gpk_gp_nll_grad.argtypes = [vp, vp, ci, ci, _i64, vp, vp, ci, cd, ci, vp, vp]
        lib.gpk_gp_nll_grad_dev.argtypes = [vp, vp, ci, ci, _i64, vp, vp, ci, cd, ci, vp, vp]
        lib.gpk_gp_model_fit.argtypes = [vp, vp, ci, ci, _i64, vp, vp, ci, cd, C.POINTER(vp), vp]
        lib.gpk_gp_model_from_factor.argtypes = [vp, vp, ci, ci, _i64, vp, _i64, vp, vp, C.POINTER(vp)]
        lib.gpk_gp_model_destroy.argtypes = [vp, vp]
        lib.gpk_gp_model_get_alpha.argtypes = [vp, vp, vp]
        lib.gpk_gp_model_append.argtypes = [vp, vp, vp, cd, ci, cd, vp]
        lib.gpk_gp_model_size.argtypes = [vp, vp]
        lib.gpk_gp_model_predict.argtypes = [vp, vp, vp, ci, _i64, ci, vp, vp, _i64, vp, _i64]
        lib.gpk_gp_models_mean.argtypes = [vp, vp, ci, vp, ci, _i64, vp]
        lib.gpk_gp_models_mean_var.argtypes = [vp, vp, ci, vp, ci, _i64, vp, vp]
        lib.gpk_gpukf_filter.argtypes = [vp, vp, ci, vp, ci, ci, ci, vp, vp, vp, cd, cd, cd, ci, vp, vp, vp]
        lib.gpk_gp_model_ucb.argtypes = [vp, vp, vp, ci, _i64, cd, vp, vp, _i64, vp, vp]
        lib.gpk_gp_predict.argtypes = [vp, vp, ci, ci, _i64, vp, vp, ci, _i64, vp, ci, cd, vp, vp, _i64, vp]
        lib.gpk_potrf_inv_block_dev.argtypes = [vp, vp, vp, ci, vp]
        lib.gpk_gemm_nt_dev.argtypes = [vp, ci, ci, ci, cd, vp, _i64, vp, _i64, cd, vp, _i64, ci]
        lib.gpk_gemv_dev.argtypes = [vp, ci, ci, ci, cd, vp, _i64, vp, cd, vp]
        lib.gpk_add_diag_dev.argtypes = [vp, vp, _i64, ci, cd]
        lib.gpk_sum_log_diag_dev.argtypes = [vp, vp, _i64, ci, vp, ci]
        lib.gpk_ep_fit.argtypes = [vp, vp, ci, _i64, vp, cd, ci, ci, ci, vp, vp, vp, vp, _i64, vp, vp, vp, vp]
        lib.gpk_ep_classify.argtypes = [vp, vp, ci, _i64, vp, ci, _i64, vp, vp, vp, vp, _i64, vp, vp, vp]
        lib.gpk_ep_nll_grad.argtypes = [vp, vp, ci, ci, _i64, vp, vp, cd, ci, ci, ci, ci, vp, vp, vp, vp, vp]
        lib.gpk_ep_nll_grad_batched.argtypes = [vp, ci, vp, ci, ci, _i64, _i64, vp, vp, _i64, cd, ci, ci, ci, ci, vp, vp, vp, vp,
                                                vp, vp]
        lib.gpk_ep_grad_from_factor.argtypes = [vp, vp, ci, ci, _i64, vp, vp, _i64, vp, vp, vp, _i64, ci, vp]
        lib.gpk_gp_nll_grad_batched.argtypes = [vp, ci, vp, ci, ci, _i64, _i64, vp, vp, ci, cd, ci, vp, vp, vp]
        lib.gpk_gp_nll_grad_batched_dev.argtypes = [vp, ci, vp, ci, ci, _i64, _i64, vp, vp, ci, cd, ci, vp, vp]
        lib.gpk_gp_predict_batched.argtypes = [vp, ci, vp, ci, ci, _i64, _i64, vp, vp, vp, ci, _i64, _i64, ci, cd, vp, vp, vp, vp]
        lib.gpk_debug_base_timing.argtypes = [vp, vp]
        lib.gpk_debug_ep_site_timing.argtypes = [vp, C.c_int, vp]
        lib.gpk_debug_ep_scalar.argtypes = [vp, ci, vp, ci, vp]
        lib.gpk_debug_ep_sites.argtypes = [vp, ci, vp, ci, ci, vp, vp, vp, vp, vp, vp, vp, vp]
        lib.gpk_debug_ep_apply.argtypes = [vp, vp, ci, ci, ci, ci, vp, vp, vp, vp, vp, vp]
        lib.gpk_debug_ep_site_loop.argtypes = [vp, vp, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp]
        lib.gpk_debug_ep_refactor.argtypes = [vp, vp, ci, vp, vp, vp, vp, vp]
        lib.gpk_debug_gemm.argtypes = [vp, vp, _i64, _i64, vp, _i64, _i64, vp, _i64, _i64, vp, _i64, _i64,
                                       ci, ci, ci, ci, cd, cd, ci, ci, ci]
        lib.gpk_debug_cov.argtypes = [vp, ci, vp, ci, _i64, vp, ci, _i64, ci, vp, ci, cd, vp, _i64, ci, ci, ci, _i64, _i64, _i64]
        lib.gpk_debug_grad_trace.argtypes = [vp, vp, ci, vp, ci, ci, _i64, vp, vp, ci, vp, ci, _i64, _i64]
        lib.gpk_debug_trmv.argtypes = [vp, ci, vp, ci, vp, vp, ci]
        lib.gpk_debug_colwise_dot.argtypes = [vp, vp, _i64, ci, ci, vp, vp, ci, ci, _i64, _i64, _i64]
        lib.gpk_debug_loglik.argtypes = [vp, vp, ci, ci, vp, vp, vp, ci, _i64]
        lib.gpk_mg_create.argtypes = [C.POINTER(vp), ci, vp]
        lib.gpk_mg_destroy.argtypes = [vp]
        lib.gpk_mg_last_error.argtypes = [vp]
        lib.gpk_mg_last_error.restype = C.c_char_p
        lib.gpk_mg_device_count.argtypes = [vp]
        lib.gpk_mg_set_block.argtypes = [vp, ci]
        lib.gpk_mg_potrf_solve.argtypes = [vp, vp, ci, ci, _i64, vp, vp, ci, cd, vp, vp, vp]
        lib.gpk_mg_last_seconds.argtypes = [vp]
        lib.gpk_mg_last_seconds.restype = cd
        lib.gpk_mg_last_put_bytes.argtypes = [vp]
        lib.gpk_mg_last_put_bytes.restype = C.c_int64
        _lib = lib
        return lib


class Handle:
    """One libgpk handle = one device + one stream (include/gpk.h). Not re-entrant."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self.lib = load()
        self._h = C.c_void_p()
        rc = self.lib.gpk_create(C.byref(self._h), int(device), C.c_void_p(stream) if stream else None)
        if rc != GPK_OK:
            raise GpkError(rc, f"gpk_create(device={device}) failed: no usable CUDA device "
                               f"(libgpk has no CPU fallback)")
        self.device = device

    @property
    def h(self):
        return self._h

    def check(self, rc):
        if rc == GPK_OK:
            return
        msg = self.lib.gpk_last_error(self._h).decode()
        if rc == GPK_EINVAL:
            raise IllegalArgumentError(rc, msg)
        if rc == GPK_ENOTSYM:
            raise MatrixNotSymmetricError(rc, msg)
        if rc == GPK_ENOTPD:
            raise NotPositiveDefiniteError(rc, msg, self.lib.gpk_last_info(self._h))
        raise GpkError(rc, msg)

    def launch_count(self) -> int:
        return int(self.lib.gpk_launch_count(self._h))

    def set_graph_mode(self, on):
        """CUDA-graph replay of repeated launch sequences (include/gpk.h): False / 0 eager only, True / 1 default policy,
        2 capture at the first repetition."""
        self.check(self.lib.gpk_set_graph_mode(self._h, int(on)))

    def kernel_family(self, family: int):
        """`with h.kernel_family(GPK_KERNEL_CO2): ...` -- how the (D, theta) arguments of the enclosed calls are read
        (include/gpk.h); the handle goes back to its previous family afterwards."""
        return _FamilyScope(self, int(family))

    def synchronize(self):
        self.check(self.lib.gpk_synchronize(self._h))

    def close(self):
        if self._h:
            self.lib.gpk_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _FamilyScope:
    def __init__(self, handle, family):
        self.h, self.family = handle, family

    def __enter__(self):
        self.prev = self.h.lib.gpk_get_kernel_family(self.h._h)
        self.h.check(self.h.lib.gpk_set_kernel_family(self.h._h, self.family))
        return self.h

    def __exit__(self, *exc):
        self.h.lib.gpk_set_kernel_family(self.h._h, self.prev)
        return False


_default = {}


def default_handle(device: int = 0) -> Handle:
    """Process-wide handle per device (the Scala objects are singletons too, spring-context.xml)."""
    if device not in _default:
        _default[device] = Handle(device)
    return _default[device]


def fmat(a) -> np.ndarray:
    """Column-major float64 view/copy: the Breeze DenseMatrix layout expected by the ABI."""
    a = np.asarray(a, dtype=np.float64)
    if a.ndim == 2 and not a.flags.f_contiguous:
        a = np.asfortranarray(a)
    elif a.ndim == 1:
        a = np.ascontiguousarray(a)
    return a


def ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)
