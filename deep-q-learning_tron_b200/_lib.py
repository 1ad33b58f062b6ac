"""ctypes binding of libtron_b200.so (the C ABI in include/tron_b200.h).

Fails loudly: a missing library or a non-zero status raises; nothing here computes on the CPU.
"""
import ctypes as C
import os

from . import _abi as abi

_HERE = os.path.dirname(os.path.abspath(__file__))
# TRON_B200_DEBUG=1 selects the range-checked build (libtron_b200_debug.so, tests only)
DEBUG = os.environ.get("TRON_B200_DEBUG", "0") == "1"
# TRON_B200_LIB=<path> loads another build of the same ABI (A/B measurements of kernel changes; tools only)
LIB_PATH = os.environ.get("TRON_B200_LIB") or os.path.join(_HERE, "libtron_b200_debug.so" if DEBUG else "libtron_b200.so")


class TronError(RuntimeError):
    pass


_lib = None

_vp, _i, _u64, _i64, _f = C.c_void_p, C.c_int, C.c_uint64, C.c_int64, C.c_float
_SIGS = {
    "tron_abi_version": (C.c_int, []),
    "tron_status_string": (C.c_char_p, [_i]),
    "tron_device_count": (C.c_int, []),
    "tron_state_bytes": (C.c_int, [_i, _i, _i, _i, C.POINTER(C.c_size_t)]),
    "tron_state_offsets": (C.c_int, [_i, _i, _i, _i, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "tron_set_option": (C.c_int, [_i, _i64]),
    "tron_cells_per_env": (C.c_int, [_i, _i]),
    "tron_enc_planes": (C.c_int, [_i]),
    "tron_dtype_size": (C.c_int, [_i]),
    "tron_build_plane_tables": (C.c_int, [_vp, _i, _vp]),
    "tron_reset": (C.c_int, [_vp, _i, _i, _i, _i, _vp, _i, _vp, _u64, _u64, _u64, _vp]),
    "tron_reset_ex": (C.c_int, [C.POINTER(abi.StepArgs), _vp, _vp]),
    "tron_step": (C.c_int, [C.POINTER(abi.StepArgs), _vp]),
    "tron_observe": (C.c_int, [C.POINTER(abi.StepArgs), _vp]),
    "tron_step_many": (C.c_int, [C.POINTER(abi.StepArgs), _vp]),
    "tron_export_grid": (C.c_int, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tron_import_grid": (C.c_int, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tron_random_actions": (C.c_int, [_vp, _i, _u64, _u64, _vp, _u64, _vp]),
    "tron_select_actions": (C.c_int, [_vp, _i, _i, _f, _vp, _u64, _u64, _vp, _u64, _vp]),
    "tron_advance_counter": (C.c_int, [_vp, _u64, _vp]),
    "tron_minimax_actions": (C.c_int, [_vp, _i, _i, _i, _i, _i, _u64, _u64, _vp, _u64, _vp, _vp, _vp, _vp]),
    "tron_pop_up": (C.c_int, [_vp, _i, _i64, _i, _vp, _i, _vp]),
    "replay_push": (C.c_int, [C.POINTER(abi.ReplayRing), _u64, _vp, _vp, _vp, _vp, _vp, _i, _i64, _vp]),
    "replay_gather": (C.c_int, [C.POINTER(abi.ReplayRing), _vp, _i64, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "replay_sample_indices": (C.c_int, [_i64, _i64, _u64, _u64, _vp, _vp]),
    "replay_sample_gather": (C.c_int, [C.POINTER(abi.ReplayRing), _i64, _i64, _u64, _u64, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "replay_frames_sample_gather": (C.c_int, [C.POINTER(abi.ReplayFrames), _i64, _i64, _i64, _u64, _u64, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "replay_states_sample_gather": (C.c_int, [C.POINTER(abi.ReplayStates), C.POINTER(abi.StepArgs), _i64, _i64, _i64, _u64, _u64, _vp, _vp, _i,
                                              _vp, _vp, _vp, _vp, _vp]),
    "tron_host_env_create": (C.c_int, [C.POINTER(_vp), C.POINTER(abi.StepArgs), _i]),
    "tron_host_env_destroy": (C.c_int, [_vp]),
    "tron_host_env_reset": (C.c_int, [_vp, _vp, _vp]),
    "tron_host_env_step": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tron_host_env_step_begin": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tron_host_env_step_wait": (C.c_int, [_vp]),
    "tron_host_copy_bandwidth": (C.c_int, [C.c_size_t, _i, _i, C.POINTER(C.c_double)]),
    "tron_debug_violations": (C.c_int, [C.POINTER(C.c_uint64), C.POINTER(C.c_int32)]),
    "tron_host_env_state": (_vp, [_vp]),
    "tron_host_alloc": (C.c_int, [C.POINTER(_vp), C.c_size_t]),
    "tron_host_free": (C.c_int, [_vp]),
}


def load():
    """Load the shared library (once).  Raises TronError when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise TronError("%s is not built (%s); run `python __graft_entry__.py build` -- "
                            "there is no CPU fallback" % (os.path.basename(LIB_PATH), LIB_PATH))
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        if L.tron_abi_version() != abi.ABI_VERSION:
            raise TronError("ABI version mismatch: library %d, python %d" % (L.tron_abi_version(), abi.ABI_VERSION))
        _lib = L
    return _lib


def check(status, what=""):
    if status != 0:
        msg = load().tron_status_string(status).decode()
        raise TronError("%s failed: %s (status %d)" % (what or "tron_b200 call", msg, status))


def require_cuda():
    n = load().tron_device_count()
    if n <= 0:
        raise TronError("no usable CUDA device (tron_device_count=%d); tron_b200 has no CPU fallback" % n)
    return n
