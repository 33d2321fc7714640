"""ctypes binding of libidqn_b200.so (C ABI declared in include/idqn_b200.h)."""
from __future__ import annotations

import ctypes as C
import os
import threading

PKG = os.path.dirname(os.path.abspath(__file__))

OK, EINVAL, ECUDA, ERANGE, EASSERT, ENOMEM = 0, -1, -2, -3, -4, -5
ARCH_FC, ARCH_CNN, ARCH_IMPALA = 0, 1, 2
ONLINE, TARGET, MU, NU, GRAD = 0, 1, 2, 3, 4
F_NO_GRAPH, F_SIMT_ONLY, F_KEEP_GRADS, F_NO_IMG, F_NO_PDL, F_PARTITION, F_OLD_WGRAD, F_NO_FORK, F_NO_DEFER, F_SLOW_APPLY = 1, 2, 4, 8, 16, 32, 64, 128, 256, 512
F_TIMELINE = 1024
F_CHAIN = 2048
MAX_FEATURES = 8
MAX_ACTIONS = 32  # HEAD_MAXA of csrc/net.cu


class LibraryError(RuntimeError):
    """libidqn_b200.so is missing / unloadable, or a CUDA call inside it failed."""


class Config(C.Structure):
    _fields_ = [
        ("arch", C.c_int32), ("obs", C.c_int32 * 3), ("n_actions", C.c_int32), ("n_heads", C.c_int32),
        ("n_features", C.c_int32), ("features", C.c_int32 * MAX_FEATURES), ("batch_size", C.c_int32),
        ("learning_rate", C.c_float), ("adam_eps", C.c_float), ("gamma_n", C.c_float),
        ("device", C.c_int32), ("flags", C.c_int32),
    ]


# every symbol include/idqn_b200.h declares: name -> (restype, argtypes)
_P, _I, _I64 = C.c_void_p, C.c_int, C.c_int64
SYMBOLS = {
    "idqn_last_error": (C.c_char_p, []),
    "idqn_version": (_I, []),
    "idqn_create": (_I, [C.POINTER(Config), C.POINTER(_P)]),
    "idqn_destroy": (_I, [_P]),
    "idqn_arena_stride": (_I64, [_P]),
    "idqn_leaf_count": (_I, [_P]),
    "idqn_leaf_info": (_I, [_P, _I, C.POINTER(_I64), C.POINTER(_I64), _P, C.POINTER(C.c_int32), _P]),
    "idqn_upload": (_I, [_P, _I, _I, _I64, _P, _I64]),
    "idqn_download": (_I, [_P, _I, _I, _I64, _P, _I64]),
    "idqn_download_activation": (_I, [_P, _I, _I, _P, _I64]),
    "idqn_set_count": (_I, [_P, _P]),
    "idqn_get_count": (_I, [_P, _P]),
    "idqn_arena_ptr": (_P, [_P, _I]),
    "idqn_mark_planes_dirty": (_I, [_P, _I]),
    "idqn_mark_head_planes_dirty": (_I, [_P, _I, _I]),
    "idqn_stream": (_P, [_P]),
    "idqn_learn_on_batch_host": (_I, [_P, _P, _P, _I, _P, _P, _P, _P]),
    "idqn_learn_on_batch_dev": (_I, [_P, _P, _P, _I, _P, _P, _P, _P]),
    "idqn_submit_batch_host": (_I, [_P, _P, _P, _I, _P, _P, _P, C.POINTER(_I64)]),
    "idqn_wait_losses": (_I, [_P, _I64, _P]),
    "idqn_set_loss_accumulation": (_I, [_P, _I]),
    "idqn_read_cumulated_losses": (_I, [_P, _P, _I]),
    "idqn_read_td_abs": (_I, [_P, _P]),
    "idqn_write_cumulated_losses": (_I, [_P, _P]),
    "idqn_kernels_per_step": (_I, [_P]),
    "idqn_profile_step": (_I, [_P, _I, _I, _P, _P, C.POINTER(_I)]),
    "idqn_debug_timeline": (_I, [_P, _I]),
    "idqn_kernel_timeline": (_I, [_P, _P, _P, _I, C.POINTER(_I)]),
    "idqn_cta_timeline": (_I, [_P, _I, _P, _I, C.POINTER(_I)]),
    "idqn_dense_update_ctas": (_I, [_P]),
    "idqn_set_dense_update_ctas": (_I, [_P, _I]),
    "idqn_shift_params": (_I, [_P]),
    "idqn_sync_target": (_I, [_P]),
    "idqn_copy_online_to_target": (_I, [_P]),
    "idqn_peer_export_size": (_I, []),
    "idqn_peer_create": (_I, [_P, C.POINTER(_P), _P]),
    "idqn_peer_connect": (_I, [_P, _P, _P]),
    "idqn_peer_destroy": (_I, [_P]),
    "idqn_peer_sync_target": (_I, [_P]),
    "idqn_peer_shift_params": (_I, [_P]),
    "idqn_apply_host": (_I, [_P, _I, _I, _P, _I, _I, _P]),
    "idqn_best_action": (_I, [_P, _I, _I, _P, _I, C.POINTER(C.c_int32)]),
    "idqn_select_action": (_I, [_P, _P, _I, C.c_uint32, C.c_uint32, _I, C.c_float, C.POINTER(C.c_int32), _P]),
    "idqn_select_actions": (_I, [_P, _P, _I, _I, _P, _I, C.c_float, _P, _P]),
    "idqn_prng":(_I, [_I, C.c_uint32, C.c_uint32, C.c_int32, C.c_int32, _P]),
    "idqn_sumtree_create": (_I, [_I64, _I, C.POINTER(_P)]),
    "idqn_sumtree_destroy": (_I, [_P]),
    "idqn_sumtree_depth": (_I, [_P]),
    "idqn_sumtree_num_nodes": (_I64, [_P]),
    "idqn_sumtree_set": (_I, [_P, _P, _P, _I64]),
    "idqn_sumtree_get": (_I, [_P, _P, _P, _I64]),
    "idqn_sumtree_root": (_I, [_P, C.POINTER(C.c_double)]),
    "idqn_sumtree_query": (_I, [_P, _P, _P, _I64]),
    "idqn_sumtree_sample": (_I, [_P, _P, _P, _I64]),
    "idqn_sumtree_read_nodes": (_I, [_P, _P]),
    "idqn_sumtree_max_recorded": (_I, [_P, C.POINTER(C.c_double)]),
    "idqn_sumtree_set_at_max": (_I, [_P, C.c_int32]),
    "idqn_sumtree_update_from_learner": (_I, [_P, _P, _P, _I]),
    "idqn_sumtree_nodes_ptr": (_P, [_P]),
    "idqn_sumtree_write_nodes": (_I, [_P, _P, C.c_double]),
    "idqn_replay_create": (_I, [_I64, _I64, _I, C.POINTER(_P)]),
    "idqn_replay_destroy": (_I, [_P]),
    "idqn_replay_put": (_I, [_P, _I64, _P, _P, C.c_int32, C.c_double, C.c_uint8, C.c_uint8]),
    "idqn_replay_gather_host": (_I, [_P, _P, _I, _P, _P, _P, _P, _P, _P]),
    "idqn_learn_from_replay": (_I, [_P, _P, _P, _I, _I, _P]),
    "idqn_replay_create_frames": (_I, [_I64, _I64, _I, _I, _I64, _I, C.POINTER(_P)]),
    "idqn_replay_put_frame": (_I, [_P, _I64, _P]),
    "idqn_replay_put_element": (_I, [_P, _I64, _P, C.c_int32, C.c_double, C.c_uint8, C.c_uint8]),
    "idqn_replay_grow_frames": (_I, [_P, _I64, _I64, _I64]),
    "idqn_replay_read_frames": (_I, [_P, _I64, _I64, _P]),
    "idqn_replay_write_frames": (_I, [_P, _I64, _I64, _P]),
    "idqn_replay_read_slots": (_I, [_P, _I64, _I64, _P, _P, _P, _P, _P, _P]),
    "idqn_replay_write_slots": (_I, [_P, _I64, _I64, _P, _P, _P, _P, _P, _P]),
    "idqn_replay_digest": (_I, [_P, _I64, _I64, _I64, _P]),
    "idqn_replay_stream": (_P, [_P]),
}

_lock = threading.Lock()
_lib = None


def library_path() -> str:
    return os.environ.get("IDQN_B200_LIB", os.path.join(PKG, "libidqn_b200.so"))


def lib() -> C.CDLL:
    """Load (once) and return the bound library.  Raises LibraryError if it is absent — there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = library_path()
        if not os.path.exists(path):
            raise LibraryError(
                f"{path} not found. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(needs nvcc); idqn_b200 has no CPU or eager fallback.")
        try:
            handle = C.CDLL(path)
        except OSError as e:  # pragma: no cover
            raise LibraryError(f"cannot load {path}: {e}") from e
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
        return _lib


def last_error() -> str:
    msg = lib().idqn_last_error()
    return msg.decode() if msg else ""


def check(rc: int) -> None:
    """Map C status codes onto the exception types the reference raises at the same places."""
    if rc == OK:
        return
    msg = last_error()
    if rc == ERANGE:
        raise ValueError(msg)  # sum_tree.py:73-74
    if rc == EASSERT:
        raise AssertionError(msg)  # sum_tree.py:12,30-31,81
    if rc == EINVAL:
        raise ValueError(msg)
    if rc == ENOMEM:
        raise MemoryError(msg)
    raise LibraryError(msg)


def ptr(a):
    """void* of a C-contiguous numpy array (caller keeps it alive)."""
    return a.ctypes.data_as(C.c_void_p)
