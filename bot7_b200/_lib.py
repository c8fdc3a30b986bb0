"""ctypes binding of libbot7_b200.so -- exactly the symbols include/bot7_b200.h declares.

The LuaJIT-FFI glue in lua/bot7_b200/ffi.lua binds the same symbols with the same signatures; this
module is its Python twin, used because no Lua runtime exists in this image.  There is no CPU
fallback: if the shared library is missing the import of any product module fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BOT7_B200_LIB") or os.path.join(_HERE, "libbot7_b200.so")

KERNEL_ARDSE, KERNEL_MATERN52 = 0, 1
SCORE_EI, SCORE_CB = 0, 1
BOUND_LOWER, BOUND_UPPER = 0, 1
FIT_PREDICT, FIT_LOGML_ONLY, FIT_DEFER = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_TANH = 0, 1, 2
PATH_FP64_DMMA, PATH_INT8_OZAKI = 0, 1
STAGES = ("sobol", "kbuild", "potrf", "trtri", "kstar", "posterior", "score", "blr")

_p = C.c_void_p
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_lp = C.POINTER(C.c_int64)
_i, _l, _d = C.c_int, C.c_int64, C.c_double

# name -> (restype, argtypes); kept in the order of include/bot7_b200.h
SIGNATURES = {
    "b7_version": (_i, []),
    "b7_last_error": (C.c_char_p, []),
    "b7_init": (_i, [_i, C.POINTER(_p)]),
    "b7_shutdown": (None, [_p]),
    "b7_device_count": (_i, []),
    "b7_sync": (_i, [_p]),
    "b7_set_profiling": (_i, [_p, _i]),
    "b7_reset_stage_timers": (_i, [_p]),
    "b7_last_stage_ms": (_i, [_p, _i, _dp, _lp]),
    "b7_set_posterior_path": (_i, [_p, _i]),
    "b7_get_posterior_path": (_i, [_p]),
    "b7_timer_begin": (_i, [_p]),
    "b7_timer_end": (_i, [_p, _dp]),
    "b7_launch_count": (_l, [_p]),
    "b7_sobol_directions": (_i, [_i, C.POINTER(C.c_uint32)]),
    "b7_sobol_generate": (_i, [_p, _i, _l, _l, _dp, _dp, _dp, C.POINTER(_p)]),
    "b7_grid_from_host": (_i, [_p, _dp, _l, _i, C.POINTER(_p)]),
    "b7_grid_read": (_i, [_p, _l, _l, _dp]),
    "b7_grid_size": (_l, [_p]),
    "b7_grid_rows": (_l, [_p]),
    "b7_grid_dims": (_i, [_p]),
    "b7_grid_remove": (_i, [_p, _l, _dp]),
    "b7_grid_original_index": (_i, [_p, _l, _lp]),
    "b7_grid_free": (None, [_p]),
    "b7_gp_fit": (_i, [_p, _i, _dp, _dp, _i, _i, _dp, _i, _i, _i, _i, C.POINTER(_p), _ip, _dp, _dp]),
    "b7_gp_refit": (_i, [_p, _dp, _i, _ip, _dp, _dp]),
    "b7_gp_num_draws": (_i, [_p]),
    "b7_gp_num_obs": (_i, [_p]),
    "b7_gp_predict": (_i, [_p, _i, _dp, _l, _dp, _dp]),
    "b7_gp_device_ptr": (_i, [_p, _i, C.POINTER(_p), _lp]),
    "b7_gp_padded_n": (_i, [_p]),
    "b7_gp_read_factor": (_i, [_p, _i, _dp]),
    "b7_gp_fit_range": (_i, [_p, _i, _i, _ip, _dp, _dp]),
    "b7_gp_invert_range": (_i, [_p, _i, _i]),
    "b7_gp_mark_ready": (_i, [_p]),
    "b7_gp_free": (None, [_p]),
    "b7_acq_score": (_i, [_p, _p, _i, _d, _i, _d, _d, _dp, _lp, _lp, _dp, _lp]),
    "b7_acq_score_range": (_i, [_p, _p, _l, _l, _i, _d, _i, _d, _d, _dp, _lp, _dp, _lp]),
    "b7_score_moments": (_i, [_p, _i, _dp, _dp, _i, _l, _d, _i, _d, _d, _dp, _lp, _dp, _lp]),
    "b7_mlp_features": (_i, [_p, _p, _i, _ip, C.POINTER(_dp), C.POINTER(_dp), _i, C.POINTER(_p)]),
    "b7_mlp_features_act": (_i, [_p, _p, _i, _ip, C.POINTER(_dp), C.POINTER(_dp), _ip, C.POINTER(_p)]),
    "b7_blr_fit": (_i, [_p, _dp, _dp, _i, _i, _dp, _i, C.POINTER(_p), _ip]),
    "b7_blr_refit": (_i, [_p, _dp, _i, _ip, _dp]),
    "b7_blr_num_draws": (_i, [_p]),
    "b7_blr_predict": (_i, [_p, _i, _dp, _l, _dp, _dp]),
    "b7_blr_score": (_i, [_p, _p, _i, _d, _i, _d, _d, _dp, _lp, _lp, _dp, _lp]),
    "b7_dngo_score": (_i, [_p, _p, _i, _ip, C.POINTER(_dp), C.POINTER(_dp), _i, _i, _d, _i, _d, _d, _dp, _lp, _lp, _dp, _lp]),
    "b7_dngo_score_act": (_i, [_p, _p, _i, _ip, C.POINTER(_dp), C.POINTER(_dp), _ip, _i, _d, _i, _d, _d, _dp, _lp, _lp, _dp, _lp]),
    "b7_blr_free": (None, [_p]),
    "b7_comm_init_all": (_i, [_i, _ip, C.POINTER(_p)]),
    "b7_comm_unique_id": (_i, [C.c_char_p]),
    "b7_comm_init_rank": (_i, [_i, C.c_char_p, _i, _i, C.POINTER(_p)]),
    "b7_comm_world": (_i, [_p]),
    "b7_comm_local_count": (_i, [_p]),
    "b7_comm_first_rank": (_i, [_p]),
    "b7_comm_ctx": (_p, [_p, _i]),
    "b7_comm_free": (None, [_p]),
    "b7_shard_range": (_i, [_l, _i, _i, _lp, _lp]),
    "b7_sobol_generate_sharded": (_i, [_p, _i, _l, _l, _dp, _dp, C.POINTER(_p)]),
    "b7_grid_from_host_sharded": (_i, [_p, _dp, _l, _i, C.POINTER(_p)]),
    "b7_grid_remove_sharded": (_i, [_p, C.POINTER(_p), _l, _dp]),
    "b7_gp_fit_sharded": (_i, [_p, _i, _dp, _dp, _i, _i, _dp, _i, _i, _i, C.POINTER(_p), _ip, _dp, _dp, _dp]),
    "b7_acq_score_multi": (_i, [_p, C.POINTER(_p), C.POINTER(_p), _i, _d, _i, _d, _d, _dp, _lp, _lp, _dp, _lp]),
    "b7_blr_fit_multi": (_i, [_p, _dp, _dp, _i, _i, _dp, _i, C.POINTER(_p), _ip]),
    "b7_dngo_score_multi": (_i, [_p, C.POINTER(_p), C.POINTER(_p), _i, _ip, C.POINTER(_dp), C.POINTER(_dp), _i, _i, _d, _i, _d, _d, _dp,
                                 _lp, _lp, _dp, _lp]),
    "b7_dngo_score_multi_act": (_i, [_p, C.POINTER(_p), C.POINTER(_p), _i, _ip, C.POINTER(_dp), C.POINTER(_dp), _ip, _i, _d, _i, _d, _d,
                                     _dp, _lp, _lp, _dp, _lp]),
}


class B7Error(RuntimeError):
    pass


def load_library(path: str = LIB_PATH) -> C.CDLL:
    if not os.path.exists(path):
        raise B7Error(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  bot7_b200 has no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError here = header/library drift
        fn.restype = res
        fn.argtypes = args
    return lib


_LIB = None


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        _LIB = load_library()
    return _LIB


def check(rc: int, what: str = "") -> int:
    if rc < 0:
        raise B7Error(f"{what}: {lib().b7_last_error().decode()} (rc={rc})")
    return rc


def as_f64(a, shape=None) -> np.ndarray:
    """Contiguous fp64 view/copy (the Lua glue calls tensor:contiguous():double())."""
    arr = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        arr = arr.reshape(shape)
    return arr


def dptr(a: np.ndarray | None):
    return None if a is None else a.ctypes.data_as(_dp)


class Context:
    """One CUDA context handle per (process, device).  b7_init fails without a GPU."""

    _default = {}

    def __init__(self, device: int = 0):
        self.handle = _p()
        check(lib().b7_init(device, C.byref(self.handle)), "b7_init")
        self.device = device

    @classmethod
    def default(cls, device: int | None = None) -> "Context":
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        if device not in cls._default:
            cls._default[device] = cls(device)
        return cls._default[device]

    def close(self):
        if self.handle:
            lib().b7_shutdown(self.handle)
            self.handle = _p()

    def sync(self):
        check(lib().b7_sync(self.handle), "b7_sync")

    def set_profiling(self, on: bool):
        check(lib().b7_set_profiling(self.handle, int(on)))

    def reset_timers(self):
        check(lib().b7_reset_stage_timers(self.handle))

    def stage_times(self) -> dict:
        out = {}
        for k, name in enumerate(STAGES):
            ms, n = _d(0.0), _l(0)
            check(lib().b7_last_stage_ms(self.handle, k, C.byref(ms), C.byref(n)))
            out[name] = (ms.value, n.value)
        return out

    def set_posterior_path(self, path: int):
        check(lib().b7_set_posterior_path(self.handle, int(path)), "b7_set_posterior_path")

    def posterior_path(self) -> int:
        return int(lib().b7_get_posterior_path(self.handle))

    def timer_begin(self):
        check(lib().b7_timer_begin(self.handle), "b7_timer_begin")

    def timer_end(self) -> float:
        ms = _d(0.0)
        check(lib().b7_timer_end(self.handle, C.byref(ms)), "b7_timer_end")
        return ms.value

    def launch_count(self) -> int:
        return int(lib().b7_launch_count(self.handle))
