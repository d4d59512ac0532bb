"""Host-side mirror of the bevy_ggrs plugin surface for the hot path.

Same names and argument meaning as the reference (src/lib.rs, src/snapshot/rollback_app.rs,
src/schedule_systems.rs) so that a bevy_ggrs user — and the parity tests — read the same:

    app = App(engine)
    app.add_plugins(GgrsPlugin())
    app.insert_resource(RollbackFrameRate(60))
    app.add_systems(ReadInputs, read_local_inputs)
    t = app.rollback_component_with_clone("Transform", 40)
    app.checksum_component(t, byte_offset=0, byte_len=12, assert_finite=True)
    app.add_systems(GgrsSchedule, System(BGR_SYS_PARTICLES_UPDATE, [t, v]))
    app.insert_resource(Session.SyncTest(session))
    app.add_observer(SyncTestMismatch, on_mismatch)
    app.update()

Differences forced by the C ABI (documented in INTEGRATION.md):
  * components are registered by (name, size_of::<T>()) and the per-element hasher is a byte
    range instead of a Rust closure;
  * GgrsSchedule systems are compiled-in GPU systems named by id, or the game's own written as CUDA source
    (``CudaSystem``);
  * the "World" is the engine: columns live in HBM, the ring of snapshots too.

``backend`` is any object with the ``bevy_ggrs_b200.engine.Engine`` method surface.  This
module is pure host logic: it never touches the GPU or the oracle itself.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Callable, Dict, List, Optional, Sequence

from . import capi
from .host_components import HostComponents
from .session import (ADVANCE, LOAD, SAVE, GgrsError, MismatchedChecksum, P2PTraceSession, Request,
                      SyncTestSession)

DEFAULT_FPS = 60  # lib.rs:58


# ---- schedule labels (lib.rs:73-74, :148-149) ----
class GgrsSchedule:
    pass


class ReadInputs:
    pass


class Startup:
    pass


# ---- resources ----
@dataclass
class RollbackFrameRate:  # time.rs:19-26
    fps: int = DEFAULT_FPS


@dataclass
class LocalInputs:  # lib.rs:140-141
    inputs: Dict[int, int]


@dataclass
class LocalPlayers:  # lib.rs:144-145
    handles: List[int] = field(default_factory=list)


@dataclass
class SyncTestMismatch:  # lib.rs:131-137
    current_frame: int
    mismatched_frames: List[int]


class Session:  # lib.rs:79-86
    SYNCTEST, P2P, SPECTATOR = "SyncTest", "P2P", "Spectator"

    def __init__(self, kind: str, inner):
        self.kind = kind
        self.inner = inner

    @classmethod
    def SyncTest(cls, s: SyncTestSession) -> "Session":
        return cls(cls.SYNCTEST, s)

    @classmethod
    def P2PTrace(cls, s: P2PTraceSession) -> "Session":
        return cls(cls.P2P, s)


@dataclass
class System:
    """A compiled-in GgrsSchedule system: id + the columns it binds + scalar parameters."""
    system: int
    columns: Sequence[int]
    params: Sequence[int] = ()


@dataclass
class CudaSystem:
    """A GgrsSchedule system of the game's own: ``BGR_SYSTEM_FN void name(const bgr_sys_ctx&, bgr_commands&, A&, ...)``
    in ``source``, one parameter per column of ``columns``, compiled into the registration's kernel at build
    (``bgr_add_user_system``)."""
    name: str
    source: str
    columns: Sequence[int]
    params: Sequence[int] = ()


@dataclass
class ResourceSystem:
    """A GgrsSchedule system that only touches host-side resources (e.g. box_game's increase_frame_system,
    box_game.rs:146-148): ``fn(resources: dict[str, bytearray])``.  Resources are a few bytes and not
    data-parallel, so they stay on the host (SURVEY.md §2 row 10); the shim rolls them back per frame and XORs
    their checksum parts into the engine's checksum."""
    fn: Callable


class GgrsPlugin:  # lib.rs:198-258
    def build(self, app: "App") -> None:
        app._ggrs = True


class App:
    """Mirror of ``bevy::App`` restricted to what the rollback hot path touches."""

    MANUAL_DURATION_NS = 16_666_667  # Duration::from_secs_f64(1.0 / 60.0), tests/common/mod.rs:47-49

    def __init__(self, backend):
        self.world = backend
        self._ggrs = False
        self._built = False
        self._session: Optional[Session] = None
        self._frame_rate = RollbackFrameRate()
        self._read_inputs: List[Callable[["App"], None]] = []
        self._startup: List[Callable[["App"], None]] = []
        self._observers: List[Callable[[SyncTestMismatch], None]] = []
        self._local_inputs: Optional[LocalInputs] = None
        self.local_players = LocalPlayers()
        # FixedTimestepData (lib.rs:98-114)
        self._accumulator_ns = 0
        self._run_slow = False
        self._first_update = True
        self.last_checksums: List[tuple] = []
        self.ticks = 0
        # host-side resources (rollback_resource_with_copy / checksum_resource_with_hash)
        self.resources: Dict[str, bytearray] = {}
        self._res_registered: List[str] = []
        self._res_checksummed: List[str] = []
        self._res_systems: List[Callable] = []
        self._res_store: Dict[int, Dict[str, bytes]] = {}
        self._res_frame = 0
        # host-side side table for rollback components that are not plain bytes (Sprite: particles.rs:191)
        self.host_components = HostComponents(backend)

    # ---- App ----
    def add_plugins(self, plugin) -> "App":
        plugin.build(self)
        return self

    def remove_resource(self, kind) -> "App":
        """`world.remove_resource::<Session<T>>()`: the next update takes the session-less branch."""
        if kind is Session:
            self._session = None
        else:
            raise TypeError(f"unsupported resource {kind!r}")
        return self

    def insert_resource(self, res) -> "App":
        if isinstance(res, Session):
            self._session = res
        elif isinstance(res, RollbackFrameRate):
            self._frame_rate = res
        elif isinstance(res, LocalInputs):
            self._local_inputs = res
        else:
            raise TypeError(f"unsupported resource {type(res).__name__}")
        return self

    def add_systems(self, schedule, system) -> "App":
        if schedule is GgrsSchedule:
            if isinstance(system, ResourceSystem):
                self._res_systems.append(system.fn)
                return self
            if isinstance(system, CudaSystem):
                self.world.add_user_system(system.name, system.source, list(system.columns), list(system.params))
                return self
            assert isinstance(system, System), "GgrsSchedule systems are GPU systems (System, CudaSystem) or ResourceSystems"
            self.world.add_system(system.system, list(system.columns), list(system.params))
        elif schedule is ReadInputs:
            self._read_inputs.append(system)
        elif schedule is Startup:
            self._startup.append(system)
        else:
            raise TypeError("unknown schedule label")
        return self

    def add_observer(self, event_type, fn) -> "App":
        assert event_type is SyncTestMismatch
        self._observers.append(fn)
        return self

    # ---- RollbackApp (rollback_app.rs:31-248) ----
    def rollback_component_with_copy(self, type_name: str, size_of: int) -> int:
        return self.world.rollback_component(type_name, size_of, capi.BGR_STRATEGY_COPY)

    def rollback_component_with_clone(self, type_name: str, size_of: Optional[int] = None, clone=None):
        """``size_of`` bytes of plain data -> an HBM column (returns its index).  ``size_of=None``: the type is Clone but
        not plain bytes (``Sprite`` holds an ``Arc`` handle, particles.rs:191) -> it stays on the host in the side table
        (host_components.py) and is rolled back there by the same request vectors; returns the ``HostColumn``."""
        if size_of is None:
            return self.host_components.register(type_name, **({"clone": clone} if clone else {}))
        return self.world.rollback_component(type_name, size_of, capi.BGR_STRATEGY_CLONE)

    def rollback_optional_component_with_copy(self, type_name: str, size_of: int) -> int:
        """A component single entities may lose / regain inside the rollback window: the ``Option<&mut S::Target>``
        match of ``ComponentSnapshotPlugin::load`` (component_snapshot.rs:99-115).  ``world.remove_component`` /
        ``world.insert_component`` are the ``commands.entity(e).remove::<T>()`` / ``.insert(t)`` of code outside
        ``GgrsSchedule``."""
        return self.world.rollback_component(type_name, size_of, capi.BGR_STRATEGY_COPY | capi.BGR_STRATEGY_OPTIONAL)

    def checksum_component(self, column: int, byte_offset: int, byte_len: int, assert_finite: bool = False) -> "App":
        self.world.checksum_component(column, byte_offset, byte_len,
                                      capi.BGR_HASH_FLAG_ASSERT_FINITE_F32 if assert_finite else 0)
        return self

    def checksum_component_with_hash(self, column: int) -> "App":
        return self.checksum_component(column, 0, self.world.elem_bytes[column])

    def rollback_resource_with_copy(self, type_name: str, initial: Optional[bytes] = None) -> "App":  # rollback_app.rs:171-176
        """``initial=None`` registers a resource that is absent for now: the snapshot stores ``None`` for it
        (GgrsResourceSnapshots = GgrsSnapshots<R, Option<As>>, mod.rs:87) and a Load re-inserts / removes it."""
        self._res_registered.append(type_name)
        if initial is not None:
            self.resources[type_name] = bytearray(initial)
        return self

    rollback_resource_with_clone = rollback_resource_with_copy

    def checksum_resource_with_hash(self, type_name: str) -> "App":  # rollback_app.rs:213-218
        self._res_checksummed.append(type_name)
        return self

    # ---- frame resources ----
    def rollback_frame_count(self) -> int:
        return self.world.rollback_frame_count()

    def confirmed_frame_count(self) -> int:
        return self.world.confirmed_frame_count()

    # ---- one Bevy frame ----
    def _finish(self) -> None:
        if not self._built:
            self.world.build()
            self._built = True
            for s in self._startup:
                s(self)

    def update(self) -> None:
        self._finish()
        # bevy Time<Real>: the first update has zero delta, later ones the manual duration
        delta = 0 if self._first_update else self.MANUAL_DURATION_NS
        self._first_update = False
        self.run_ggrs_schedules(delta)

    def step(self) -> None:
        """Exactly one GGRS tick regardless of the accumulator (benches)."""
        self._finish()
        self._tick()

    # ---- run_ggrs_schedules (schedule_systems.rs:19-83) ----
    def run_ggrs_schedules(self, delta_ns: int) -> None:
        fps = self._frame_rate.fps
        fps_delta = (1_000_000_000 * 11 // (fps * 10)) if self._run_slow else (1_000_000_000 // fps)
        self._accumulator_ns += delta_ns
        while self._accumulator_ns >= fps_delta:
            self._accumulator_ns -= fps_delta
            if self._session is None:
                # "No session has been started yet, reset time data and snapshots" (schedule_systems.rs:70-79)
                self._accumulator_ns = 0
                self._run_slow = False
                self.local_players = LocalPlayers([])
                self.world.reset_session()  # RollbackFrameCount(0), ConfirmedFrameCount(-1), MaxPredictionWindow(8)
                return
            self._tick()

    def _tick(self) -> None:
        sess = self._session
        inner = sess.inner
        self.local_players = LocalPlayers(list(range(inner.num_players())))
        # world.run_schedule(ReadInputs) (:89 / :144)
        self._local_inputs = None
        for s in self._read_inputs:
            s(self)
        if self._local_inputs is None:
            raise RuntimeError("No local player inputs found. Did you insert systems into the ReadInputs schedule?")
        for handle, value in self._local_inputs.inputs.items():
            inner.add_local_input(handle, value)
        try:
            requests = inner.advance_frame()
        except MismatchedChecksum as e:  # :104-115
            ev = SyncTestMismatch(e.current_frame, e.mismatched_frames)
            for obs in self._observers:
                obs(ev)
            return
        except GgrsError:
            return
        self.handle_requests(requests)
        self.ticks += 1

    # ---- handle_requests (schedule_systems.rs:170-289) ----
    def handle_requests(self, requests: Sequence[Request]) -> None:
        inner = self._session.inner
        checksums = self.world.handle_requests(inner.info(), requests)
        if self._res_registered:
            checksums = self._handle_resource_requests(requests, checksums)
        if self.host_components.columns:
            self.host_components.handle_requests(requests)
        # cell.save(frame, None, checksum) (:236)
        for frame, cs in checksums:
            inner.save_cell(frame, cs)
        self.last_checksums = checksums

    # host-side half of handle_requests for resources (resource_snapshot.rs:65-93, resource_checksum.rs:63-82):
    # the same request vector, replayed on a few bytes of host state; parts are XORed into the engine's
    # checksum exactly like ChecksumPlugin::update folds every ChecksumPart (checksum.rs:88-99).
    def _handle_resource_requests(self, requests, checksums):
        import ctypes as C
        lib = capi.load_library()
        out, k = [], 0
        for r in requests:
            if r.kind == SAVE:  # resource_snapshot.rs:65-73: Some(clone) or None
                self._res_store[self._res_frame] = {n: (bytes(self.resources[n]) if n in self.resources else None)
                                                    for n in self._res_registered}
                part = 0
                for name in self._res_checksummed:  # resource_checksum.rs:63-82 (the resource must exist)
                    b = bytes(self.resources[name])
                    part ^= lib.bgr_seahash(C.create_string_buffer(b, len(b)), len(b))
                frame, cs = checksums[k]
                out.append((frame, cs ^ part))
                k += 1
            elif r.kind == LOAD:  # resource_snapshot.rs:77-93: update / insert / remove
                self._res_frame = r.frame
                for n, v in self._res_store[r.frame].items():
                    if v is None:
                        self.resources.pop(n, None)
                    else:
                        self.resources[n] = bytearray(v)
            else:
                self._res_frame += 1
                for fn in self._res_systems:
                    if fn.__code__.co_argcount >= 2:
                        fn(self.resources, self._res_frame)   # (resources, RollbackFrameCount)
                    else:
                        fn(self.resources)
        alive = set(self.world.snapshot_frames())
        self._res_store = {f: v for f, v in self._res_store.items() if f in alive}
        return out
