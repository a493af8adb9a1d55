"""ctypes binding of libcolosseum_b200.so (include/colosseum_b200.h).

There is no CPU fallback: if the CUDA library is missing, cannot be loaded, or no sm_100 device is
present, every use raises.  The library is built in-tree by ``colosseumrl_b200/build.py`` (nvcc,
``-gencode arch=compute_100a,code=sm_100a``).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcolosseum_b200.so")

NSTAT = 32
ERR_ARG, ERR_CUDA, ERR_UNSUPPORTED = 1, 2, 3     # CRL_ERR_* of include/colosseum_b200.h
STAT_ROWS = 256
FLAG_AUTO_RESET = 1
FLAG_COMPACT_RESULT = 2      # crl_tron_step: 4-byte result record
FLAG_COMPACT2_RESULT = 8     # crl_tron_step: 2-byte result record
FLAG_PACKED_ACTIONS = 4      # crl_tron_step: uint8[B] actions, 2 bits per player

_vp, _i64, _i32, _u64, _u32, _int = C.c_void_p, C.c_int64, C.c_int32, C.c_uint64, C.c_uint32, C.c_int

# symbol -> (restype, argtypes); mirrors include/colosseum_b200.h one to one
SIGNATURES = {
    "crl_version": (_int, []),
    "crl_last_error": (C.c_char_p, []),
    "crl_init": (_int, [_int]),
    "crl_philox_words": (_int, [_vp, _u64, _u64, _u32, _u32, _i64, _vp]),
    "crl_stats_reduce": (_int, [_vp, _vp, _int, _vp]),
    "crl_host_graph_launch": (_int, [_vp, _vp, _vp]),
    "crl_host_graph_launch_wait": (_int, [_vp, _vp, _vp, _vp]),
    "crl_host_event_wait": (_int, [_vp]),
    "crl_tron_state_bytes": (_i64, [_int, _int, _i64]),
    "crl_tron_action_stride": (_int, [_int, _int]),
    "crl_tron_result_bytes": (_int, [_int, _int]),
    "crl_tron_policy_random_wide": (_int, [_vp, _u64, _u64, _u32, _i64, _vp]),
    "crl_tron_start_positions": (_int, [_int, _int, C.POINTER(_i32), C.POINTER(_i32)]),
    "crl_tron_reset": (_int, [_vp, _vp, _i64, _int, _int, _vp]),
    "crl_tron_start_positions_at": (_int, [_int, _int, _int, _int, C.POINTER(_i32), C.POINTER(_i32)]),
    "crl_tron_reset_at": (_int, [_vp, _vp, _i64, _int, _int, _int, _int, _vp]),
    "crl_tron_start_positions_spawns": (_int, [_int, _int, _int, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32)]),
    "crl_tron_reset_spawns": (_int, [_vp, _vp, _i64, _int, _int, _int, C.POINTER(_i32), _vp]),
    "crl_tron_step_spawns": (_int, [_vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _int, _int, C.POINTER(_i32), _vp]),
    "crl_tron_step": (_int, [_vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _int, _vp]),
    "crl_tron_policy_random": (_int, [_vp, _u64, _u64, _u32, _i64, _vp]),
    "crl_tron_rollout": (_int, [_vp, _vp, _vp, _u64, _u64, _u32, _int, _i64, _int, _int, _vp]),
    "crl_tron_observe": (_int, [_vp, _int, _vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _vp]),
    "crl_tron_ranking": (_int, [_vp, _vp, _i64, _int, _int, _vp]),
    "crl_tron_pack": (_int, [_vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _vp]),
    "crl_ttt_cells": (_int, [_int]),
    "crl_ttt_lines": (_int, [_int, C.POINTER(_u32), _int]),
    "crl_ttt_reset": (_int, [_vp, _vp, _i64, _int, _vp]),
    "crl_ttt_step": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _vp]),
    "crl_ttt_valid_actions": (_int, [_vp, _vp, _i64, _int, _vp]),
    "crl_ttt_policy_random": (_int, [_vp, _vp, _u64, _u64, _u32, _i64, _int, _int, _vp]),
    "crl_ttt_rollout": (_int, [_vp, _vp, _vp, _u64, _u64, _u32, _int, _i64, _int, _vp]),
    "crl_ttt_observe": (_int, [_vp, _int, _vp, _vp, _vp, _i64, _int, _vp]),
    "crl_ttt_pack": (_int, [_vp, _vp, _vp, _vp, _i64, _int, _vp]),
    "crl_blokus_state_bytes": (_i64, [_i64]),
    "crl_blokus_reset": (_int, [_vp, _vp, _i64, _vp]),
    "crl_blokus_legal": (_int, [_vp, _int, _vp, _vp, _i32, _vp, _i64, _int, _vp]),
    "crl_blokus_is_valid": (_int, [_vp, _int, _vp, _vp, _i64, _int, _vp]),
    "crl_blokus_step": (_int, [_vp, _vp, _vp, _vp, _vp, _i64, _int, _vp]),
    "crl_blokus_policy_random": (_int, [_vp, _vp, _i32, _vp, _u64, _u64, _u32, _i64, _vp]),
    "crl_blokus_rollout": (_int, [_vp, _vp, _vp, _u64, _u64, _u32, _int, _i64, _vp]),
    "crl_blokus_pick": (_int, [_vp, _vp, _i32, _vp, _vp, _i64, _vp]),
    "crl_blokus_observe": (_int, [_vp, _int, _vp, _vp, _vp, _vp, _i64, _vp]),
    "crl_blokus_pack": (_int, [_vp, _vp, _vp, _vp, _vp, _i64, _vp]),
}

# ... and of the companion header include/colosseum_b200_tron_policy.h (device-side Tron opponents)
TRON_POLICY_SIGNATURES = {
    "crl_tron_policy_avoid": (_int, [_vp, _vp, _int, _int, _u64, _u64, _u32, _i64, _int, _int, _int, _int,
                                     C.POINTER(_i32), _vp]),
    "crl_tron_rollout_avoid": (_int, [_vp, _vp, _vp, _u64, _u64, _u32, _int, _i64, _int, _int, _int, _int, _int,
                                      C.POINTER(_i32), _vp]),
}

# ... and of the companion header include/colosseum_b200_learner.h (one learner against device-side random opponents)
LEARNER_SIGNATURES = {
    "crl_ttt_advance": (_int, [_vp, _vp, _int, _vp, _vp, _vp, _u64, _u64, _u32, _i64, _int, _vp]),
    "crl_blokus_advance": (_int, [_vp, _vp, _int, _vp, _vp, _u64, _u64, _u32, _i64, _vp]),
}

# ... and of the companion header include/colosseum_b200_placement.h (Blokus placements: masks, placement -> action id)
PLACEMENT_SIGNATURES = {
    "crl_blokus_placement_mask": (_int, [_vp, _int, _int, _vp, _vp, _i64, _int, _vp]),
    "crl_blokus_placement_to_action": (_int, [_vp, _int, _int, _vp, _vp, _i64, _int, _vp]),
    "crl_blokus_shape_table": (_int, [_vp, _vp, _vp, _vp]),
}


class CrlError(RuntimeError):
    pass


def declare(lib):
    """Attach restype/argtypes for every exported symbol; raises if one is missing."""
    tables = (SIGNATURES, TRON_POLICY_SIGNATURES, LEARNER_SIGNATURES, PLACEMENT_SIGNATURES)
    for name, (res, args) in [item for table in tables for item in table.items()]:
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    return lib


_lib = None


def load():
    """Load the CUDA library (no device needed yet). Raises CrlError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CrlError("%s not found: build it with `python -m colosseumrl_b200.build` "
                           "(there is no CPU fallback)" % LIB_PATH)
        _lib = declare(C.CDLL(LIB_PATH))
    return _lib


def check(rc, lib=None):
    if rc != 0:
        lib = lib or load()
        raise CrlError("libcolosseum_b200 error %d: %s" % (rc, lib.crl_last_error().decode()))


_inited = set()


def init(device_index: int):
    lib = load()
    if device_index not in _inited:
        check(lib.crl_init(device_index), lib)
        _inited.add(device_index)
    return lib
