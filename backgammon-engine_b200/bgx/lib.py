"""ctypes binding of libbgx.so (include/bgx.h).  Loads the in-tree build only.

There is no fallback of any kind: if the library is missing, `load()` raises, and the
batched entry points raise `BgxError` when no CUDA device is present (BGX_E_NO_DEVICE).
"""
import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(_PKG, "lib", "libbgx.so")

OK, E_INVALID, E_NO_DEVICE, E_CUDA, E_CAPACITY, E_STATE = 0, -1, -2, -3, -4, -5
FIRST_ROLLOFF, FIRST_PARITY = 0, 1
ROLLOUT_STRATIFY, ROLLOUT_MAX_PLIES = 1, 4096
NPARAMS, NPARAMS_PADDED = 25601, 25604


class BgxError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libbgx error {code}: {msg}")
        self.code = code


class Stats(C.Structure):
    _fields_ = [("plies", C.c_int64), ("sequences", C.c_int64), ("scored", C.c_int64),
                ("games_finished", C.c_int64), ("p1_wins", C.c_int64), ("truncated", C.c_int64),
                ("td_steps", C.c_int64), ("td_sq_error", C.c_double), ("tree_edges", C.c_int64),
                ("td_live_rows", C.c_int64), ("td_lazy_row_steps", C.c_int64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_vp = C.c_void_p
_i64 = C.c_int64
_SIGNATURES = {
    # section 1
    "bgx_last_error": (C.c_char_p, []),
    "bgx_abi_version": (C.c_int, []),
    "bgx_legal_moves": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int, C.POINTER(C.c_int)]),
    "bgx_try_move": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "bgx_move_error_string": (C.c_char_p, [C.c_int]),
    "bgx_game_over": (C.c_int, [_vp, C.POINTER(C.c_int)]),
    "bgx_turn_sequences": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _i64, _vp, _vp, _vp, C.POINTER(_i64)]),
    # section 2
    "bgx_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "bgx_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "bgx_destroy": (C.c_int, [_vp]),
    "bgx_set_stream": (C.c_int, [_vp, _vp]),
    "bgx_synchronize": (C.c_int, [_vp]),
    "bgx_set_weights": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "bgx_get_weights": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    # section 3
    "bgx_enumerate_summary": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "bgx_enumerate_summary_host": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "bgx_enumerate": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    "bgx_enumerate_count": (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "bgx_enumerate_host": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, C.POINTER(_i64)]),
    "bgx_encode": (C.c_int, [_vp, _vp, _i64, _vp]),
    "bgx_encode_host": (C.c_int, [_vp, _vp, _i64, _vp]),
    "bgx_evaluate": (C.c_int, [_vp, _vp, _i64, _vp]),
    "bgx_evaluate_host": (C.c_int, [_vp, _vp, _i64, _vp]),
    "bgx_select_moves": (C.c_int, [_vp, _vp, _i64, C.c_float, C.c_uint64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bgx_select_moves_host": (C.c_int, [_vp, _vp, _i64, C.c_float, C.c_uint64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bgx_select_moves_2ply": (C.c_int, [_vp, _vp, _i64, C.c_int32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bgx_select_moves_2ply_host": (C.c_int, [_vp, _vp, _i64, C.c_int32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bgx_rollout": (C.c_int, [_vp, _vp, _i64, C.c_int32, C.c_int32, C.c_uint64, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bgx_rollout_host": (C.c_int, [_vp, _vp, _i64, C.c_int32, C.c_int32, C.c_uint64, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bgx_rollout_vr": (C.c_int, [_vp, _vp, _i64, C.c_int32, C.c_int32, C.c_uint64, C.c_int, C.c_int32] + [_vp] * 9),
    "bgx_rollout_vr_host": (C.c_int, [_vp, _vp, _i64, C.c_int32, C.c_int32, C.c_uint64, C.c_int, C.c_int32] + [_vp] * 9),
    "bgx_select_moves_host_async":(C.c_int, [_vp, C.c_int, _vp, _i64, C.c_float, C.c_uint64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bgx_play_ply_host_async": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, _i64, C.c_float, C.c_uint64, C.c_uint64, _vp, _vp, _vp, _vp]),
    "bgx_play_ply_restart_host_async": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, _i64, C.c_int, _i64, C.c_float, C.c_uint64, C.c_uint64, _vp, _vp, _vp, _vp]),
    "bgx_lane_wait": (C.c_int, [_vp, C.c_int]),
    "bgx_advance": (C.c_int, [_vp, _vp, _vp, _i64, C.c_uint64, C.c_int32, _vp, _vp]),
    "bgx_set_host_threads": (C.c_int, [C.c_int]),
    "bgx_advance_host": (C.c_int, [_vp, _vp, _i64, C.c_uint64, _vp, _vp, _vp]),
    # section 4
    "bgx_selfplay_init": (C.c_int, [_vp, _i64, _i64, _i64, C.c_uint64, C.c_int, C.c_int32]),
    "bgx_selfplay_record_chosen": (C.c_int, [_vp, C.c_int]),
    "bgx_selfplay_step": (C.c_int, [_vp, C.c_int32, C.c_float, C.POINTER(Stats)]),
    "bgx_selfplay_round": (C.c_int, [_vp, C.c_float, C.POINTER(Stats)]),
    "bgx_selfplay_next_round": (C.c_int, [_vp]),
    "bgx_selfplay_read": (C.c_int, [_vp, _vp, _vp, _vp]),
    "bgx_export_trajectory": (C.c_int, [_vp, _i64, C.c_int32, _vp, _vp, C.POINTER(C.c_int32)]),
    "bgx_selfplay_sample": (C.c_int, [_vp, C.c_int32, C.c_uint64, _vp]),
    "bgx_selfplay_sample_host": (C.c_int, [_vp, C.c_int32, C.c_uint64, _vp]),
    # section 5
    "bgx_td_replay": (C.c_int, [_vp, C.c_double, C.c_double, _vp, C.POINTER(Stats)]),
    "bgx_td_replay_scheduled": (C.c_int, [_vp, _i64, _vp, C.POINTER(Stats)]),
    "bgx_apply_delta": (C.c_int, [_vp, _vp, C.c_float]),
    "bgx_td_round_host": (C.c_int, [_vp, C.c_double, C.c_double, C.c_float, _vp, C.POINTER(Stats)]),
    "bgx_td_replay_host": (C.c_int, [_vp, _vp, C.c_int32, C.c_int, C.c_double, C.c_double, _vp, _vp, _vp, _vp, _vp]),
    "bgx_allreduce_delta": (C.c_int, [_vp, _vp, _vp]),
    "bgx_nccl_load": (C.c_int, [C.c_char_p]),
    "bgx_nccl_unique_id": (C.c_int, [_vp]),
    "bgx_nccl_comm_init": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.POINTER(_vp)]),
    "bgx_nccl_comm_destroy": (C.c_int, [_vp]),
    # section 6
    "bgx_launch_count": (C.c_int, [_vp, C.POINTER(_i64)]),
    "bgx_last_kernel_ms": (C.c_int, [_vp, C.POINTER(C.c_float)]),
    "bgx_kernel_config": (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "bgx_sfu_monotone": (C.c_int, [_vp, C.POINTER(_i64), C.POINTER(_i64)]),
    "bgx_set_option": (C.c_int, [_vp, C.c_char_p, _i64]),
    "bgx_twoply_stage_ms": (C.c_int, [_vp, _vp]),
    "bgx_td_profile": (C.c_int, [_vp, C.c_int, _vp]),
    "bgx_device_props": (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(_i64)]),
}

_lib = None


def load(path=None):
    """dlopen the in-tree libbgx.so; raise if it was not built (run __graft_entry__.build())."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise FileNotFoundError(f"{path} not found: build it with `python __graft_entry__.py build` "
                                "(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here == header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def exported_symbols():
    return sorted(_SIGNATURES)


def check(rc):
    if rc != OK:
        raise BgxError(rc, load().bgx_last_error().decode(errors="replace"))


def ptr(a):
    """Raw address of a numpy array, a torch tensor (host or CUDA), an int, or None."""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        assert a.flags["C_CONTIGUOUS"], "buffers must be C-contiguous"
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        assert a.is_contiguous(), "tensors must be contiguous"
        return a.data_ptr()
    raise TypeError(type(a))
