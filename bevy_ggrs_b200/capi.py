"""ctypes view of ``include/bevy_ggrs_b200.h`` (the C-ABI drop-in boundary).

The shared library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a) as
``bevy_ggrs_b200/libbevy_ggrs_b200.so``.  There is NO CPU fallback: if the library is missing
``load_library()`` raises, and ``bgr_engine_create`` fails with BGR_ERR_CUDA on a box without
a usable GPU.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Iterable, List, Optional, Sequence

BGR_ABI_VERSION = 1
BGR_MAX_PLAYERS = 8
BGR_MAX_REQUESTS = 80
BGR_MAX_CHECKSUM_COLUMNS = 6

# bgr_status
BGR_OK, BGR_ERR_INVALID_ARGUMENT, BGR_ERR_STATE, BGR_ERR_CUDA, BGR_ERR_NO_SNAPSHOT, \
    BGR_ERR_MISSING_RESOURCE, BGR_ERR_NON_FINITE, BGR_ERR_CAPACITY, BGR_ERR_UNSUPPORTED = range(9)
# bgr_strategy
BGR_STRATEGY_COPY, BGR_STRATEGY_CLONE = 0, 1
BGR_STRATEGY_OPTIONAL = 0x100
BGR_MAX_OPTIONAL_COLUMNS = 7
# bgr_hash_kind
BGR_HASH_NONE, BGR_HASH_BYTES = 0, 1
BGR_HASH_FLAG_ASSERT_FINITE_F32 = 1
# bgr_system
BGR_SYS_PARTICLES_UPDATE = 1
BGR_SYS_PARTICLES_DESPAWN = 2
BGR_SYS_BOX_MOVE = 3
BGR_SYS_U32_ADD = 4
BGR_SYS_U32_SATSUB_DESPAWN = 5
BGR_SYS_U32_STORE_CALL_COUNT = 6
BGR_SYS_PARTICLES_SPAWN = 7
BGR_SYS_DESPAWN_ON_INPUT = 8
BGR_INPUT_SPAWN = 0x10
# bgr_request_kind
BGR_REQ_SAVE, BGR_REQ_LOAD, BGR_REQ_ADVANCE = 0, 1, 2
# bgr_session_kind
BGR_SESSION_NONE, BGR_SESSION_SYNCTEST, BGR_SESSION_P2P, BGR_SESSION_SPECTATOR = 0, 1, 2, 3
# bgr_config.flags
BGR_CFG_FORCE_STEPWISE = 1
BGR_CFG_SHARDED = 2
BGR_CFG_SKIP_UNCHANGED_PLANES = 4


class bgr_request(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("frame", C.c_int32), ("n_players", C.c_uint32),
                ("inputs", C.c_uint8 * BGR_MAX_PLAYERS), ("status", C.c_uint8 * BGR_MAX_PLAYERS)]


class bgr_session_info(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("max_prediction", C.c_uint32), ("check_distance", C.c_uint32),
                ("confirmed_frame", C.c_int32)]


class bgr_checksum(C.Structure):
    _fields_ = [("frame", C.c_int32), ("has_checksum", C.c_uint32), ("lo", C.c_uint64), ("hi", C.c_uint64)]


class bgr_partial(C.Structure):
    _fields_ = [("frame", C.c_int32), ("n_columns", C.c_uint32), ("active", C.c_uint64), ("total", C.c_uint64),
                ("xor_", C.c_uint64 * BGR_MAX_CHECKSUM_COLUMNS)]


class bgr_config(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("device", C.c_int32), ("max_entities", C.c_uint32),
                ("max_depth", C.c_uint32), ("fps", C.c_uint32), ("flags", C.c_uint32),
                ("order_base", C.c_uint64), ("stream", C.c_void_p)]


u32p = C.POINTER(C.c_uint32)
i32p = C.POINTER(C.c_int32)
u64p = C.POINTER(C.c_uint64)
u8p = C.POINTER(C.c_uint8)

# name -> (restype, argtypes); every symbol declared in include/bevy_ggrs_b200.h
PROTOTYPES = {
    "bgr_abi_version": (C.c_uint32, []),
    "bgr_last_error": (C.c_char_p, []),
    "bgr_engine_create": (C.c_int, [C.POINTER(bgr_config), C.POINTER(C.c_void_p)]),
    "bgr_engine_destroy": (None, [C.c_void_p]),
    "bgr_rollback_component": (C.c_int, [C.c_void_p, C.c_char_p, C.c_uint32, C.c_uint32, u32p]),
    "bgr_checksum_component": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]),
    "bgr_add_system": (C.c_int, [C.c_void_p, C.c_uint32, u32p, C.c_uint32, u32p, C.c_uint32]),
    "bgr_add_user_system": (C.c_int, [C.c_void_p, C.c_char_p, C.c_char_p, u32p, C.c_uint32, u32p, C.c_uint32]),
    "bgr_build": (C.c_int, [C.c_void_p]),
    "bgr_run_startup_system": (C.c_int, [C.c_void_p, C.c_uint32]),
    "bgr_spawn": (C.c_int, [C.c_void_p, C.c_uint32, u32p]),
    "bgr_despawn": (C.c_int, [C.c_void_p, C.c_uint32]),
    "bgr_row_count": (C.c_int, [C.c_void_p, u32p]),
    "bgr_active_count": (C.c_int, [C.c_void_p, u64p]),
    "bgr_write_component": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32]),
    "bgr_read_component": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32]),
    "bgr_read_alive": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "bgr_remove_component": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32]),
    "bgr_insert_component": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "bgr_has_component": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]),
    "bgr_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "bgr_host_free": (C.c_int, [C.c_void_p]),
    "bgr_download_begin": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, u32p]),
    "bgr_download_wait": (C.c_int, [C.c_void_p, C.c_uint32]),
    "bgr_rollback_frame_count": (C.c_int, [C.c_void_p, i32p]),
    "bgr_set_rollback_frame_count": (C.c_int, [C.c_void_p, C.c_int32]),
    "bgr_confirmed_frame_count": (C.c_int, [C.c_void_p, i32p]),
    "bgr_max_prediction_window": (C.c_int, [C.c_void_p, u32p]),
    "bgr_set_depth": (C.c_int, [C.c_void_p, C.c_uint32]),
    "bgr_confirm": (C.c_int, [C.c_void_p, C.c_int32]),
    "bgr_snapshot_frames": (C.c_int, [C.c_void_p, i32p, C.c_uint32, u32p]),
    "bgr_peek": (C.c_int, [C.c_void_p, C.c_int32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32,
                           C.c_void_p, i32p]),
    "bgr_save_world": (C.c_int, [C.c_void_p, C.POINTER(bgr_checksum)]),
    "bgr_load_world": (C.c_int, [C.c_void_p]),
    "bgr_advance_world": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]),
    "bgr_handle_requests": (C.c_int, [C.c_void_p, C.POINTER(bgr_session_info), C.POINTER(bgr_request), C.c_uint32,
                                      C.POINTER(bgr_checksum), C.c_uint32, u32p]),
    "bgr_submit_requests": (C.c_int, [C.c_void_p, C.POINTER(bgr_session_info), C.POINTER(bgr_request), C.c_uint32]),
    "bgr_collect": (C.c_int, [C.c_void_p, C.POINTER(bgr_checksum), C.c_uint32, u32p]),
    "bgr_last_partials": (C.c_int, [C.c_void_p, C.POINTER(bgr_partial), C.c_uint32, u32p]),
    "bgr_fold_partials": (C.c_int, [C.POINTER(bgr_partial), C.POINTER(bgr_checksum)]),
    "bgr_collect_partials": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, u32p]),
    "bgr_fold_partials_n": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p]),
    "bgr_seahash": (C.c_uint64, [C.c_void_p, C.c_uint64]),
    "bgr_ggrs_time_delta_bits": (C.c_uint32, [C.c_uint32, C.c_int32]),
    "bgr_particle_rng_stream": (C.c_int, [C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_float, C.c_float]),
    "bgr_splitmix64_stream": (C.c_int, [C.c_uint64, C.c_uint32, C.c_void_p]),
    "bgr_launch_count": (C.c_int, [C.c_void_p, u64p]),
    "bgr_slot_bytes": (C.c_int, [C.c_void_p, u64p]),
    "bgr_last_path": (C.c_int, [C.c_void_p, u32p]),
    "bgr_generic_specialised": (C.c_int, [C.c_void_p, u32p]),
    "bgr_synchronize": (C.c_int, [C.c_void_p]),
    "bgr_stream": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "bgr_trace_enable": (C.c_int, [C.c_void_p, C.c_uint32]),
    "bgr_trace_read": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, u32p]),
    "bgr_host_profile": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32]),
    "bgr_reset_session": (C.c_int, [C.c_void_p]),
    "bgr_shard_group_join": (C.c_int, [C.c_void_p, C.c_char_p, C.c_uint32, C.c_uint32, C.c_uint32]),
    "bgr_shard_group_leave": (C.c_int, [C.c_void_p]),
    "bgr_group_join": (C.c_void_p, [C.c_char_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]),
    "bgr_group_leave": (None, [C.c_void_p]),
    "bgr_group_publish": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32]),
    "bgr_group_collect": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(bgr_checksum), C.c_uint32, u32p]),
    "bgr_ring_create": (C.c_void_p, [C.c_uint32]),
    "bgr_ring_destroy": (None, [C.c_void_p]),
    "bgr_ring_depth": (C.c_uint32, [C.c_void_p]),
    "bgr_ring_set_depth": (C.c_int, [C.c_void_p, C.c_uint32]),
    "bgr_ring_push": (C.c_int, [C.c_void_p, C.c_int32, u32p]),
    "bgr_ring_confirm": (C.c_int, [C.c_void_p, C.c_int32]),
    "bgr_ring_rollback": (C.c_int, [C.c_void_p, C.c_int32, u32p]),
    "bgr_ring_get": (C.c_int, [C.c_void_p, u32p]),
    "bgr_ring_peek": (C.c_int, [C.c_void_p, C.c_int32, u32p, i32p]),
}

_LIB: Optional[C.CDLL] = None


def library_path() -> str:
    # BGR_LIBRARY: an alternative build of the same library (tuning experiments only)
    return os.environ.get("BGR_LIBRARY") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libbevy_ggrs_b200.so")


def load_library() -> C.CDLL:
    """dlopen the in-tree C-ABI library and bind every declared symbol.  Fails loudly."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} is missing: the CUDA extension was not built (run `python -c 'import __graft_entry__ as g; "
            f"g.build()'`).  bevy_ggrs_b200 has no CPU fallback.")
    lib = C.CDLL(path)
    for name, (restype, argtypes) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.bgr_abi_version() != BGR_ABI_VERSION:
        raise RuntimeError("bevy_ggrs_b200 ABI version mismatch")
    _LIB = lib
    return lib


class BgrError(RuntimeError):
    """A non-zero bgr_status; ``.status`` holds the code, the text is what the reference would panic with."""

    def __init__(self, status: int, text: str):
        super().__init__(text)
        self.status = status


def make_requests(requests: Iterable) -> "C.Array[bgr_request]":
    """``session.Request`` objects -> a contiguous bgr_request array."""
    reqs = list(requests)
    arr = (bgr_request * max(1, len(reqs)))()
    for i, r in enumerate(reqs):
        arr[i].kind = r.kind
        arr[i].frame = r.frame
        ins = list(r.inputs)
        st = list(r.status) if r.status else [0] * len(ins)
        arr[i].n_players = len(ins)
        for j, v in enumerate(ins[:BGR_MAX_PLAYERS]):
            arr[i].inputs[j] = v & 0xFF
            arr[i].status[j] = st[j] if j < len(st) else 0
    return arr


def make_session_info(info: Sequence[int]) -> bgr_session_info:
    kind, maxp, cd, cf = info
    return bgr_session_info(kind, maxp, cd, cf)
