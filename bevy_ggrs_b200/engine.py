"""Thin object wrapper over the C ABI (``include/bevy_ggrs_b200.h``): numpy in, numpy out.

Every method is one C-ABI call.  Nothing here computes: columns, snapshots, checksums and the
re-simulation all happen in the CUDA library.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import capi
from .capi import BgrError


class Engine:
    def __init__(self, max_entities: int, max_depth: int = 9, fps: int = 60, device: int = 0, flags: int = 0,
                 order_base: int = 0, stream: Optional[int] = None):
        self._lib = capi.load_library()
        cfg = capi.bgr_config(capi.BGR_ABI_VERSION, device, max_entities, max_depth, fps, flags, order_base,
                              C.c_void_p(stream) if stream else None)
        handle = C.c_void_p()
        self._h = None
        self._check(self._lib.bgr_engine_create(C.byref(cfg), C.byref(handle)))
        self._h = handle
        self.elem_bytes: List[int] = []
        self.max_entities = max_entities
        self._pinned: List[C.c_void_p] = []

    # ---- plumbing ----
    def _check(self, status: int) -> None:
        if status != capi.BGR_OK:
            raise BgrError(status, self._lib.bgr_last_error().decode("utf-8", "replace"))

    def close(self) -> None:
        if self._h is not None:
            self._lib.bgr_engine_destroy(self._h)  # waits for every download in flight
            self._h = None
            for p in self._pinned:
                self._lib.bgr_host_free(p)
            self._pinned = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- registration (RollbackApp) ----
    def rollback_component(self, name: str, elem_bytes: int, strategy: int = capi.BGR_STRATEGY_COPY) -> int:
        col = C.c_uint32()
        self._check(self._lib.bgr_rollback_component(self._h, name.encode(), elem_bytes, strategy, C.byref(col)))
        self.elem_bytes.append(elem_bytes)
        return col.value

    def checksum_component(self, col: int, byte_offset: int, byte_len: int, flags: int = 0) -> None:
        self._check(self._lib.bgr_checksum_component(self._h, col, capi.BGR_HASH_BYTES, byte_offset, byte_len, flags))

    def add_system(self, system: int, cols: Sequence[int], params: Sequence[int] = ()) -> None:
        ca = (C.c_uint32 * max(1, len(cols)))(*cols)
        pa = (C.c_uint32 * max(1, len(params)))(*params)
        self._check(self._lib.bgr_add_system(self._h, system, ca, len(cols), pa, len(params)))

    def add_user_system(self, name: str, source: str, cols: Sequence[int], params: Sequence[int] = ()) -> None:
        """A GgrsSchedule system of the game's own, as CUDA source (contract: bgr_add_user_system in the header)."""
        ca = (C.c_uint32 * max(1, len(cols)))(*cols)
        pa = (C.c_uint32 * max(1, len(params)))(*params)
        self._check(self._lib.bgr_add_user_system(self._h, name.encode(), source.encode(), ca, len(cols), pa, len(params)))

    def build(self) -> None:
        self._check(self._lib.bgr_build(self._h))

    def run_startup_system(self, system: int) -> None:
        self._check(self._lib.bgr_run_startup_system(self._h, system))

    # ---- entities ----
    def spawn(self, count: int) -> int:
        first = C.c_uint32()
        self._check(self._lib.bgr_spawn(self._h, count, C.byref(first)))
        return first.value

    def despawn(self, row: int) -> None:
        self._check(self._lib.bgr_despawn(self._h, row))

    def row_count(self) -> int:
        v = C.c_uint32()
        self._check(self._lib.bgr_row_count(self._h, C.byref(v)))
        return v.value

    def active_count(self) -> int:
        v = C.c_uint64()
        self._check(self._lib.bgr_active_count(self._h, C.byref(v)))
        return v.value

    def write_component(self, col: int, first_row: int, values: np.ndarray) -> None:
        eb = self.elem_bytes[col]
        a = np.ascontiguousarray(values).view(np.uint8).reshape(-1, eb)
        self._check(self._lib.bgr_write_component(self._h, col, first_row, a.shape[0], a.ctypes.data, eb))

    def read_component(self, col: int, first_row: int, count: int) -> np.ndarray:
        eb = self.elem_bytes[col]
        out = np.zeros((count, eb), dtype=np.uint8)
        self._check(self._lib.bgr_read_component(self._h, col, first_row, count, out.ctypes.data, eb))
        return out

    def read_alive(self, first_row: int, count: int) -> np.ndarray:
        out = np.zeros(count, dtype=np.uint8)
        self._check(self._lib.bgr_read_alive(self._h, first_row, count, out.ctypes.data))
        return out

    # ---- per-entity presence of BGR_STRATEGY_OPTIONAL columns ----
    def remove_component(self, col: int, row: int) -> None:
        self._check(self._lib.bgr_remove_component(self._h, col, row))

    def insert_component(self, col: int, row: int, value) -> None:
        a = np.ascontiguousarray(value).view(np.uint8).reshape(-1)
        assert a.size == self.elem_bytes[col]
        self._check(self._lib.bgr_insert_component(self._h, col, row, a.ctypes.data))

    def has_component(self, col: int, first_row: int, count: int) -> np.ndarray:
        out = np.zeros(count, dtype=np.uint8)
        self._check(self._lib.bgr_has_component(self._h, col, first_row, count, out.ctypes.data))
        return out

    # ---- asynchronous mirror download (bgr_download_begin / bgr_download_wait) ----
    def host_alloc(self, count: int, byte_len: int) -> np.ndarray:
        """Page-locked (count, byte_len) u8 array for download_begin; freed with the engine."""
        p = C.c_void_p()
        self._check(self._lib.bgr_host_alloc(count * byte_len, C.byref(p)))
        self._pinned.append(p)
        buf = (C.c_uint8 * max(1, count * byte_len)).from_address(p.value)
        return np.frombuffer(buf, dtype=np.uint8, count=count * byte_len).reshape(count, byte_len)

    def download_begin(self, col: int, byte_offset: int, byte_len: int, first_row: int, count: int, dst: np.ndarray) -> int:
        assert dst.dtype == np.uint8 and dst.flags.c_contiguous and dst.size >= count * byte_len
        t = C.c_uint32()
        self._check(self._lib.bgr_download_begin(self._h, col, byte_offset, byte_len, first_row, count, dst.ctypes.data,
                                                 C.byref(t)))
        return t.value

    def download_wait(self, ticket: int) -> None:
        self._check(self._lib.bgr_download_wait(self._h, ticket))

    # ---- frame resources ----
    def rollback_frame_count(self) -> int:
        v = C.c_int32()
        self._check(self._lib.bgr_rollback_frame_count(self._h, C.byref(v)))
        return v.value

    def set_rollback_frame_count(self, frame: int) -> None:
        self._check(self._lib.bgr_set_rollback_frame_count(self._h, frame))

    def confirmed_frame_count(self) -> int:
        v = C.c_int32()
        self._check(self._lib.bgr_confirmed_frame_count(self._h, C.byref(v)))
        return v.value

    def max_prediction_window(self) -> int:
        v = C.c_uint32()
        self._check(self._lib.bgr_max_prediction_window(self._h, C.byref(v)))
        return v.value

    # ---- ring ----
    def set_depth(self, depth: int) -> None:
        self._check(self._lib.bgr_set_depth(self._h, depth))

    def confirm(self, frame: int) -> None:
        self._check(self._lib.bgr_confirm(self._h, frame))

    def snapshot_frames(self) -> List[int]:
        buf = (C.c_int32 * 128)()
        n = C.c_uint32()
        self._check(self._lib.bgr_snapshot_frames(self._h, buf, 128, C.byref(n)))
        return [buf[i] for i in range(n.value)]

    def peek(self, frame: int, col: int, first_row: int, count: int) -> Optional[Tuple[np.ndarray, np.ndarray]]:
        eb = self.elem_bytes[col]
        out = np.zeros((count, eb), dtype=np.uint8)
        alive = np.zeros(count, dtype=np.uint8)
        found = C.c_int32()
        self._check(self._lib.bgr_peek(self._h, frame, col, first_row, count, out.ctypes.data, eb,
                                       alive.ctypes.data, C.byref(found)))
        return (out, alive) if found.value else None

    # ---- schedules ----
    def save_world(self) -> Tuple[int, int]:
        cs = capi.bgr_checksum()
        self._check(self._lib.bgr_save_world(self._h, C.byref(cs)))
        return cs.frame, (cs.hi << 64) | cs.lo

    def load_world(self) -> None:
        self._check(self._lib.bgr_load_world(self._h))

    def advance_world(self, inputs: Sequence[int] = (), status: Sequence[int] = ()) -> None:
        n = len(inputs)
        ia = (C.c_uint8 * capi.BGR_MAX_PLAYERS)(*[v & 0xFF for v in inputs])
        sa = (C.c_uint8 * capi.BGR_MAX_PLAYERS)(*list(status)[:n])
        self._check(self._lib.bgr_advance_world(self._h, ia, sa, n))

    # ---- the hot loop ----
    def handle_requests(self, session_info: Sequence[int], requests) -> List[Tuple[int, int]]:
        reqs = list(requests)
        arr = capi.make_requests(reqs)
        info = capi.make_session_info(session_info)
        out = (capi.bgr_checksum * capi.BGR_MAX_REQUESTS)()
        n = C.c_uint32()
        self._check(self._lib.bgr_handle_requests(self._h, C.byref(info), arr, len(reqs), out,
                                                  capi.BGR_MAX_REQUESTS, C.byref(n)))
        return [(out[i].frame, (out[i].hi << 64) | out[i].lo) for i in range(n.value)]

    def submit_requests(self, session_info: Sequence[int], requests) -> None:
        reqs = list(requests)
        arr = capi.make_requests(reqs)
        info = capi.make_session_info(session_info)
        self._check(self._lib.bgr_submit_requests(self._h, C.byref(info), arr, len(reqs)))

    def submit_prepared(self, info: "capi.bgr_session_info", arr, n: int) -> None:
        """submit with pre-built ctypes buffers (bench inner loop: no Python marshalling in the timed region)."""
        self._check(self._lib.bgr_submit_requests(self._h, C.byref(info), arr, n))

    def collect(self) -> List[Tuple[int, int]]:
        out = (capi.bgr_checksum * capi.BGR_MAX_REQUESTS)()
        n = C.c_uint32()
        self._check(self._lib.bgr_collect(self._h, out, capi.BGR_MAX_REQUESTS, C.byref(n)))
        return [(out[i].frame, (out[i].hi << 64) | out[i].lo) for i in range(n.value)]

    def last_partials(self) -> List["capi.bgr_partial"]:
        out = (capi.bgr_partial * capi.BGR_MAX_REQUESTS)()
        n = C.c_uint32()
        self._check(self._lib.bgr_last_partials(self._h, out, capi.BGR_MAX_REQUESTS, C.byref(n)))
        return [out[i] for i in range(n.value)]

    # ---- introspection ----
    def launch_count(self) -> int:
        v = C.c_uint64()
        self._check(self._lib.bgr_launch_count(self._h, C.byref(v)))
        return v.value

    def slot_bytes(self) -> int:
        v = C.c_uint64()
        self._check(self._lib.bgr_slot_bytes(self._h, C.byref(v)))
        return v.value

    def last_path_fused(self) -> bool:
        v = C.c_uint32()
        self._check(self._lib.bgr_last_path(self._h, C.byref(v)))
        return bool(v.value)

    def generic_specialised(self) -> bool:
        """True if bgr_build compiled this registration's own kernel (NVRTC, csrc/generic_program_jit.cuh)."""
        v = C.c_uint32()
        self._check(self._lib.bgr_generic_specialised(self._h, C.byref(v)))
        return bool(v.value)

    def synchronize(self) -> None:
        self._check(self._lib.bgr_synchronize(self._h))

    def stream(self) -> int:
        """cudaStream_t (as an int) the engine launches on — for timing events recorded by the caller."""
        p = C.c_void_p()
        self._check(self._lib.bgr_stream(self._h, C.byref(p)))
        return p.value or 0

    def reset_session(self) -> None:
        """schedule_systems.rs:70-79: no session -> RollbackFrameCount(0), ConfirmedFrameCount(-1), MaxPredictionWindow(8)."""
        self._check(self._lib.bgr_reset_session(self._h))

    # ---- device-side launch trace ----
    def trace_enable(self, capacity: int) -> None:
        self._check(self._lib.bgr_trace_enable(self._h, capacity))

    def trace_read(self, capacity: int) -> np.ndarray:
        """(n, 4) uint64 per traced fused launch, GPU globaltimer ns: first block start, last block end, results
        published, reserved."""
        out = np.zeros((capacity, 4), dtype=np.uint64)
        n = C.c_uint32()
        self._check(self._lib.bgr_trace_read(self._h, out.ctypes.data, capacity, C.byref(n)))
        return out[: n.value]

    def host_profile(self) -> dict:
        out = (C.c_uint64 * 8)()
        self._check(self._lib.bgr_host_profile(self._h, out, 8))
        return {"calls": out[0], "compile_ns": out[1], "launch_ns": out[2], "wait_ns": out[3], "fold_ns": out[4]}

    # ---- shard group (multi-GPU): cross-shard checksum fold inside the engine ----
    def shard_group_join(self, name: str, rank: int, world_size: int, timeout_ms: int = 0) -> None:
        self._check(self._lib.bgr_shard_group_join(self._h, name.encode(), rank, world_size, timeout_ms))

    def shard_group_leave(self) -> None:
        self._check(self._lib.bgr_shard_group_leave(self._h))


def fold_partials(partial: "capi.bgr_partial") -> int:
    lib = capi.load_library()
    cs = capi.bgr_checksum()
    st = lib.bgr_fold_partials(C.byref(partial), C.byref(cs))
    if st != capi.BGR_OK:
        raise BgrError(st, lib.bgr_last_error().decode())
    return (cs.hi << 64) | cs.lo


def ggrs_time_delta_bits(fps: int, frame: int) -> int:
    return capi.load_library().bgr_ggrs_time_delta_bits(fps, frame)
