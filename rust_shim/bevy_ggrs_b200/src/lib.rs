//! bevy_ggrs' rollback hot path on a B200, behind bevy_ggrs' OWN names.  SOURCE ONLY — never compiled in the build
//! image (no Rust toolchain there); the same call sequence is compiled and tested from C++ and Python
//! (bevy_ggrs_b200/host/bevy_ggrs.hpp, bevy_ggrs_b200/plugin.py).
//!
//! What a user changes in `examples/stress_tests/particles.rs`: the import, one resource, and marker impls for the
//! components whose rollback moves to the GPU — the registration calls keep the reference's names and signatures
//! (`RollbackApp`, bevy_ggrs src/snapshot/rollback_app.rs:31-133):
//!
//! ```ignore
//! use bevy_ggrs_b200::prelude::*;                          // was: use bevy_ggrs::prelude::*;
//!
//! unsafe impl GpuColumn for Transform { const BYTES: u32 = 40; }          // translation | rotation | scale
//! unsafe impl GpuColumn for Velocity  { const BYTES: u32 = 12; }
//! unsafe impl GpuColumn for Ttl       { const BYTES: u32 = 8;  }
//! impl ByteRangeHash for Velocity  { const RANGE: (u32, u32) = (0, 12); const ASSERT_FINITE_F32: bool = true; }
//! impl ByteRangeHash for Transform { const RANGE: (u32, u32) = (0, 12); const ASSERT_FINITE_F32: bool = true; }
//!
//! app.insert_resource(B200Config { max_entities: 1_000_000, max_depth: 9, device: 0 })
//!    .add_plugins(GgrsPlugin::<Config>::default())                       // unchanged call, this crate's plugin
//!    .rollback_component_with_clone::<Transform>()                       // unchanged
//!    .rollback_component_with_copy::<Velocity>()                         // unchanged
//!    .rollback_component_with_copy::<Ttl>()                              // unchanged
//!    .rollback_resource_with_clone::<ParticleRng>()                      // unchanged: resources stay host-side
//!    .checksum_component_with_hash::<Velocity>()                         // unchanged
//!    .checksum_component::<Transform>(translation_bits_hasher)           // unchanged; checked against RANGE at registration
//!    // was: .add_systems(GgrsSchedule, (update_particles, despawn_particles)) — closures cannot cross to the GPU,
//!    // the systems the hot path needs are compiled in (include/bevy_ggrs_b200.h `bgr_system`):
//!    .add_gpu_systems(&[(GpuSystem::ParticlesUpdate, &[TypeId::of::<Transform>(), TypeId::of::<Velocity>()]),
//!                       (GpuSystem::ParticlesDespawn, &[TypeId::of::<Ttl>()])])
//!    .insert_resource(Session::P2P(session));                            // unchanged
//! ```
//!
//! `Rollback`, `RollbackId`, `Session`, `GgrsSchedule`, `ReadInputs`, `LocalInputs`, `LocalPlayers`, `PlayerInputs`,
//! `RollbackFrameRate`, `RollbackFrameCount`, `ConfirmedFrameCount`, `MaxPredictionWindow`, `Checksum`,
//! `SyncTestMismatch` are bevy_ggrs' own items, re-exported.  Components registered through this crate's
//! `RollbackApp` live in HBM (the ECS copy is a mirror, see [`mirror_component`]); everything else the reference
//! snapshots on the host (resources, `Time<GgrsTime>`, user components without a `GpuColumn` impl) keeps running
//! through bevy_ggrs' own SaveWorld / LoadWorld / AdvanceWorld schedules inside [`handle_requests`].
use std::any::TypeId;
use std::ffi::{CStr, CString};

use bevy::ecs::schedule::ScheduleLabel;
use bevy::platform::collections::HashMap;
use bevy::prelude::*;
use bevy_ggrs_b200_sys as sys;
use ggrs::{Config, GgrsError, GgrsRequest, SessionState};

pub mod prelude {
    pub use super::{AddGpuSystems, B200Config, ByteRangeHash, CudaSystem, GgrsPlugin, GpuColumn, GpuSystem, RollbackApp, mirror_component};
    pub use bevy_ggrs::{
        AddRollbackCommandExtension, Checksum, ConfirmedFrameCount, GgrsConfig, GgrsSchedule, GgrsTime, LocalInputs, LocalPlayers,
        MaxPredictionWindow, PlayerInputs, ReadInputs, Rollback, RollbackFrameCount, RollbackFrameRate, RollbackId, Session, SyncTestMismatch,
    };
    pub use ggrs::{GgrsEvent as GgrsSessionEvent, PlayerType, SessionBuilder};
}
use bevy_ggrs::{
    AdvanceWorld, Checksum, ConfirmedFrameCount, GgrsSchedule, LoadWorld, LocalInputs, LocalPlayers, MaxPredictionWindow, PlayerInputs,
    ReadInputs, Rollback, RollbackFrameCount, RollbackFrameRate, SaveWorld, Session, SyncTestMismatch,
};

// ------------------------------------------------------------------------------------------------------------------
// engine handle + status -> panic
// ------------------------------------------------------------------------------------------------------------------
/// Where the rollback columns live.  Insert before `GgrsPlugin`; defaults: 1M entities, 9 frame slots, device 0.
#[derive(Resource, Clone, Copy)]
pub struct B200Config { pub max_entities: u32, pub max_depth: u32, pub device: i32 }
impl Default for B200Config { fn default() -> Self { Self { max_entities: 1 << 20, max_depth: 9, device: 0 } } }

/// The engine handle, a non-send resource (one caller thread, like the exclusive system that owns the World,
/// schedule_systems.rs:19,170).
pub struct B200Engine { raw: *mut sys::bgr_engine, built: bool }
impl Drop for B200Engine { fn drop(&mut self) { unsafe { sys::bgr_engine_destroy(self.raw) } } }

/// Non-zero status -> the panic the reference would have raised, same text
/// (e.g. "Could not rollback to 99: no snapshot at that moment could be found.", mod.rs:209-212).
fn check(status: i32) {
    if status != sys::BGR_OK {
        let text = unsafe { CStr::from_ptr(sys::bgr_last_error()) }.to_string_lossy().into_owned();
        panic!("{text}");
    }
}

// ------------------------------------------------------------------------------------------------------------------
// marker traits: which components can live in HBM, and which hashers the GPU can evaluate
// ------------------------------------------------------------------------------------------------------------------
/// A component whose rollback data is `BYTES` plain bytes at the start of the Rust value (no pointers, no Drop):
/// what `CopyStrategy` / `CloneStrategy` of a POD amount to (strategy.rs:42-83).  `BYTES` may be smaller than
/// `size_of::<Self>()` (Transform: 40 payload bytes of 48).  Unsafe: the first `BYTES` bytes must be the full state.
pub unsafe trait GpuColumn: Component { const BYTES: u32; }

/// `checksum_component::<T>(hasher)` where `hasher(t) == seahash(bytes[RANGE.0 .. RANGE.0 + RANGE.1] of t)` — what
/// `#[derive(Hash)]` produces for integer PODs and what the particles hashers do with `x.to_bits()`
/// (particles.rs:107-120, 207-222).  A closure cannot cross to the GPU; this declaration can.
pub trait ByteRangeHash: GpuColumn { const RANGE: (u32, u32); const ASSERT_FINITE_F32: bool = false; }

/// The GgrsSchedule systems with a compiled GPU twin (include/bevy_ggrs_b200.h `bgr_system`).
#[derive(Clone, Copy)]
pub enum GpuSystem { ParticlesUpdate = 1, ParticlesDespawn = 2, BoxMove = 3, ParticlesSpawn = 7 }

#[derive(Resource, Default)]
struct Columns { by_type: HashMap<TypeId, u32>, bytes: HashMap<TypeId, u32>, mirrored: Vec<(TypeId, u32, u32)> }
/// RollbackOrdered index (== engine row, rollback.rs:66-83) <-> Entity
#[derive(Resource, Default)]
struct Rows { entity_of_row: Vec<Entity>, row_of: HashMap<Entity, u32>, uploaded: u32 }

fn engine(world: &World) -> *mut sys::bgr_engine { world.non_send_resource::<B200Engine>().raw }

// ------------------------------------------------------------------------------------------------------------------
// RollbackApp — the reference's trait, same method names and signatures (rollback_app.rs:31-133, :135-248)
// ------------------------------------------------------------------------------------------------------------------
pub trait RollbackApp {
    /// rollback_app.rs:157-166.  `Type: GpuColumn` moves the column to HBM.
    fn rollback_component_with_copy<Type: Component + Copy + GpuColumn>(&mut self) -> &mut Self;
    /// rollback_app.rs:168-183
    fn rollback_component_with_clone<Type: Component + Clone + GpuColumn>(&mut self) -> &mut Self;
    /// rollback_app.rs:199-211 — the type's `Hash` must be the declared byte range (checked on probe values in debug builds)
    fn checksum_component_with_hash<Type: Component + std::hash::Hash + ByteRangeHash>(&mut self) -> &mut Self;
    /// rollback_app.rs:227-232 — same signature; `hasher` must equal the declared byte-range hash
    fn checksum_component<Type: Component + ByteRangeHash>(&mut self, hasher: for<'a> fn(&'a Type) -> u64) -> &mut Self;
    /// resources stay on the host: forwarded to bevy_ggrs' own plugins (resource_snapshot.rs, resource_checksum.rs)
    fn rollback_resource_with_copy<Type: Resource + Copy>(&mut self) -> &mut Self;
    fn rollback_resource_with_clone<Type: Resource + Clone>(&mut self) -> &mut Self;
    fn checksum_resource_with_hash<Type: Resource + std::hash::Hash>(&mut self) -> &mut Self;
}

fn register<T: GpuColumn>(app: &mut App, strategy: u32) {
    let name = CString::new(std::any::type_name::<T>()).unwrap();
    let mut col = 0u32;
    check(unsafe { sys::bgr_rollback_component(engine(app.world()), name.as_ptr(), T::BYTES, strategy, &mut col) });
    let mut cols = app.world_mut().resource_mut::<Columns>();
    cols.by_type.insert(TypeId::of::<T>(), col);
    cols.bytes.insert(TypeId::of::<T>(), T::BYTES);
}

fn register_checksum<T: ByteRangeHash>(app: &mut App) {
    let col = app.world().resource::<Columns>().by_type[&TypeId::of::<T>()];
    let flags = if T::ASSERT_FINITE_F32 { sys::BGR_HASH_FLAG_ASSERT_FINITE_F32 } else { 0 };
    check(unsafe { sys::bgr_checksum_component(engine(app.world()), col, sys::BGR_HASH_BYTES, T::RANGE.0, T::RANGE.1, flags) });
}

/// `seahash(bytes[range] of value)` through the engine's own host-side hasher (`checksum_hasher()`, mod.rs:315-317)
fn byte_range_hash<T: ByteRangeHash>(value: &T) -> u64 {
    let p = (value as *const T).cast::<u8>();
    unsafe { sys::bgr_seahash(p.add(T::RANGE.0 as usize).cast(), T::RANGE.1 as u64) }
}

impl RollbackApp for App {
    fn rollback_component_with_copy<T: Component + Copy + GpuColumn>(&mut self) -> &mut Self { register::<T>(self, sys::BGR_STRATEGY_COPY); self }
    fn rollback_component_with_clone<T: Component + Clone + GpuColumn>(&mut self) -> &mut Self { register::<T>(self, sys::BGR_STRATEGY_CLONE); self }
    fn checksum_component_with_hash<T: Component + std::hash::Hash + ByteRangeHash>(&mut self) -> &mut Self { register_checksum::<T>(self); self }
    fn checksum_component<T: Component + ByteRangeHash>(&mut self, hasher: for<'a> fn(&'a T) -> u64) -> &mut Self {
        // the closure cannot run on the GPU; it must BE the declared byte-range hash — verified on a zeroed value
        let probe: T = unsafe { core::mem::zeroed() };
        assert_eq!(hasher(&probe), byte_range_hash(&probe), "checksum_component::<{}>: the hasher is not seahash over ByteRangeHash::RANGE", std::any::type_name::<T>());
        core::mem::forget(probe);
        register_checksum::<T>(self);
        self
    }
    fn rollback_resource_with_copy<T: Resource + Copy>(&mut self) -> &mut Self { bevy_ggrs::RollbackApp::rollback_resource_with_copy::<T>(self) }
    fn rollback_resource_with_clone<T: Resource + Clone>(&mut self) -> &mut Self { bevy_ggrs::RollbackApp::rollback_resource_with_clone::<T>(self) }
    fn checksum_resource_with_hash<T: Resource + std::hash::Hash>(&mut self) -> &mut Self { bevy_ggrs::RollbackApp::checksum_resource_with_hash::<T>(self) }
}

/// Keep the ECS copy of `T` up to date for host-side readers (rendering reads `Transform`): bytes
/// [offset, offset+len) of every row are downloaded asynchronously after each tick (bgr_download_begin / _wait,
/// INTEGRATION.md "Per-tick mirror") and written into the components before `PostUpdate`.
pub fn mirror_component<T: GpuColumn>(app: &mut App, offset: u32, len: u32) -> &mut App {
    app.world_mut().resource_mut::<Columns>().mirrored.push((TypeId::of::<T>(), offset, len));
    app.add_systems(PostUpdate, mirror_into_ecs::<T>)
}

// ------------------------------------------------------------------------------------------------------------------
// GgrsPlugin — same name, same constructors (lib.rs:198-224), build = lib.rs:226-258 with the engine in place of
// SnapshotPlugin's component half
// ------------------------------------------------------------------------------------------------------------------
pub struct GgrsPlugin<C: Config> { schedule: bevy::ecs::intern::Interned<dyn ScheduleLabel>, _c: core::marker::PhantomData<C> }
impl<C: Config> Default for GgrsPlugin<C> { fn default() -> Self { Self::new(PreUpdate) } }
impl<C: Config> GgrsPlugin<C> {
    pub fn new(schedule: impl ScheduleLabel) -> Self { Self { schedule: schedule.intern(), _c: core::marker::PhantomData } }
}

#[derive(Resource, Default)]
struct FixedTimestepData { accumulator: core::time::Duration, run_slow: bool }

impl<C: Config<Input = u8>> Plugin for GgrsPlugin<C> {
    fn build(&self, app: &mut App) {
        let cfg = app.world().get_resource::<B200Config>().copied().unwrap_or_default();
        let fps = app.world().get_resource::<RollbackFrameRate>().map(|r| **r as u32).unwrap_or(60);
        let c = sys::bgr_config { abi_version: sys::BGR_ABI_VERSION, device: cfg.device, max_entities: cfg.max_entities, max_depth: cfg.max_depth,
                                  fps, flags: 0, order_base: 0, stream: core::ptr::null_mut() };
        let mut raw = core::ptr::null_mut();
        check(unsafe { sys::bgr_engine_create(&c, &mut raw) });
        app.insert_non_send_resource(B200Engine { raw, built: false })
            .init_resource::<Columns>()
            .init_resource::<Rows>()
            .init_resource::<FixedTimestepData>()
            .init_resource::<RollbackFrameCount>()
            .init_resource::<ConfirmedFrameCount>()
            .init_resource::<LocalPlayers>()
            .init_resource::<Checksum>()
            // the host-side half of SnapshotPlugin: sets, resource snapshots, Time<GgrsTime>, ChecksumPart folding
            .add_plugins((bevy_ggrs::SnapshotSetPlugin, bevy_ggrs::ChecksumPlugin, bevy_ggrs::GgrsTimePlugin))
            .add_observer(on_rollback_added)                                   // rollback.rs:40-54 -> bgr_spawn
            .add_systems(self.schedule, run_ggrs_schedules::<C>);
    }
}

/// `Rollback` on_add (rollback.rs:40-54 pushes the entity into RollbackOrdered): the entity becomes the next engine row.
fn on_rollback_added(ev: On<Add, Rollback>, mut rows: ResMut<Rows>) {
    let row = rows.entity_of_row.len() as u32;
    rows.entity_of_row.push(ev.entity);
    rows.row_of.insert(ev.entity, row);
}

/// ECS -> HBM for rows that appeared since the last tick (spawned with `Rollback` outside GgrsSchedule).
fn upload_new_rows(world: &mut World) {
    let (first, n) = { let r = world.resource::<Rows>(); (r.uploaded, r.entity_of_row.len() as u32 - r.uploaded) };
    if n == 0 { return; }
    let e = engine(world);
    if !world.non_send_resource::<B200Engine>().built {
        check(unsafe { sys::bgr_build(e) });
        world.non_send_resource_mut::<B200Engine>().built = true;
    }
    let mut base = 0u32;
    check(unsafe { sys::bgr_spawn(e, n, &mut base) });
    assert_eq!(base, first, "engine rows and RollbackOrdered indices diverged");
    let cols: Vec<(TypeId, u32, u32)> = { let c = world.resource::<Columns>(); c.by_type.iter().map(|(t, &id)| (*t, id, c.bytes[t])).collect() };
    for (ty, col, bytes) in cols {
        let Some(cid) = world.components().get_id(ty) else { continue };
        let mut stage = vec![0u8; n as usize * bytes as usize];
        for i in 0..n {
            let ent = world.resource::<Rows>().entity_of_row[(first + i) as usize];
            if let Some(ptr) = world.entity(ent).get_by_id(cid).ok() {
                unsafe { core::ptr::copy_nonoverlapping(ptr.as_ptr(), stage.as_mut_ptr().add(i as usize * bytes as usize), bytes as usize) };
            }
        }
        check(unsafe { sys::bgr_write_component(e, col, first, n, stage.as_ptr().cast(), bytes) });
    }
    world.resource_mut::<Rows>().uploaded = first + n;
}

/// HBM -> ECS for a mirrored column (runs in PostUpdate, before the renderer extracts).
fn mirror_into_ecs<T: GpuColumn>(world: &mut World) {
    let n = world.resource::<Rows>().uploaded;
    if n == 0 { return; }
    let (col, bytes) = { let c = world.resource::<Columns>(); (c.by_type[&TypeId::of::<T>()], c.bytes[&TypeId::of::<T>()]) };
    let mut stage = vec![0u8; n as usize * bytes as usize];
    let mut alive = vec![0u8; n as usize];
    let e = engine(world);
    check(unsafe { sys::bgr_read_component(e, col, 0, n, stage.as_mut_ptr().cast(), bytes) });
    check(unsafe { sys::bgr_read_alive(e, 0, n, alive.as_mut_ptr()) });
    let ents = world.resource::<Rows>().entity_of_row.clone();
    for (i, ent) in ents.iter().enumerate().take(n as usize) {
        if alive[i] == 0 { if let Ok(ec) = world.get_entity_mut(*ent) { ec.despawn(); } continue; }
        if let Some(mut t) = world.get_mut::<T>(*ent) {
            unsafe { core::ptr::copy_nonoverlapping(stage.as_ptr().add(i * bytes as usize), (&mut *t as *mut T).cast::<u8>(), bytes as usize) };
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// run_ggrs_schedules / handle_requests — schedule_systems.rs:19-289 with ONE engine call per request vector
// ------------------------------------------------------------------------------------------------------------------
fn run_ggrs_schedules<C: Config<Input = u8>>(world: &mut World) {
    let framerate: usize = **world.get_resource_or_insert_with::<RollbackFrameRate>(Default::default);
    let mut td = world.remove_resource::<FixedTimestepData>().expect("failed to extract GGRS FixedTimeStepData");
    let delta = world.resource::<Time>().delta();
    let fps_delta = if td.run_slow { core::time::Duration::from_nanos(1_000_000_000u64 * 11 / (framerate as u64 * 10)) }
                    else { core::time::Duration::from_nanos(1_000_000_000u64 / framerate as u64) };
    td.accumulator = td.accumulator.saturating_add(delta);
    if let Some(mut s) = world.get_resource_mut::<Session<C>>() {
        match &mut *s { Session::P2P(s) => s.poll_remote_clients(), Session::Spectator(s) => s.poll_remote_clients(), _ => {} }
    }
    while td.accumulator >= fps_delta {
        td.accumulator = td.accumulator.saturating_sub(fps_delta);
        upload_new_rows(world);
        match world.remove_resource::<Session<C>>() {
            Some(Session::SyncTest(mut s)) => {
                world.insert_resource(LocalPlayers((0..s.num_players()).collect()));
                world.run_schedule(ReadInputs);
                let li = world.remove_resource::<LocalInputs<C>>().expect("No local player inputs found. Did you insert systems into the ReadInputs schedule?");
                for (h, i) in li.0 { s.add_local_input(h, i).expect("All handles in local_handles should be valid"); }
                let reqs = s.advance_frame();
                let info = sys::bgr_session_info { kind: sys::BGR_SESSION_SYNCTEST, max_prediction: s.max_prediction() as u32, check_distance: s.check_distance() as u32, confirmed_frame: 0 };
                world.insert_resource(Session::SyncTest(s));
                match reqs {
                    Ok(r) => handle_requests::<C>(r, info, world),
                    Err(GgrsError::MismatchedChecksum { current_frame, mismatched_frames }) => world.trigger(SyncTestMismatch { current_frame, mismatched_frames }),
                    Err(e) => warn!("{e}"),
                }
            }
            Some(Session::P2P(mut s)) => {
                td.run_slow = s.frames_ahead() > 0;
                world.insert_resource(LocalPlayers(s.local_player_handles()));
                if s.current_state() == SessionState::Running {
                    world.run_schedule(ReadInputs);
                    let li = world.remove_resource::<LocalInputs<C>>().expect("No local player inputs found. Did you insert systems into the ReadInputs schedule?");
                    for (h, i) in li.0 { s.add_local_input(h, i).expect("All handles in local_handles should be valid"); }
                    let reqs = s.advance_frame();
                    let info = sys::bgr_session_info { kind: sys::BGR_SESSION_P2P, max_prediction: s.max_prediction() as u32, check_distance: 0, confirmed_frame: s.confirmed_frame() };
                    world.insert_resource(Session::P2P(s));
                    match reqs { Ok(r) => handle_requests::<C>(r, info, world), Err(GgrsError::PredictionThreshold) => info!("Skipping a frame: PredictionThreshold."), Err(e) => warn!("{e}") }
                } else { world.insert_resource(Session::P2P(s)); }
            }
            Some(Session::Spectator(mut s)) => {
                let reqs = (s.current_state() == SessionState::Running).then(|| s.advance_frame());
                let info = sys::bgr_session_info { kind: sys::BGR_SESSION_SPECTATOR, max_prediction: 0, check_distance: 0, confirmed_frame: 0 };
                world.insert_resource(Session::Spectator(s));
                match reqs { Some(Ok(r)) => handle_requests::<C>(r, info, world), Some(Err(GgrsError::PredictionThreshold)) => info!("P2PSpectatorSession: Waiting for input from host."), Some(Err(e)) => warn!("{e}"), None => {} }
            }
            None => {  // schedule_systems.rs:70-79
                td.accumulator = core::time::Duration::ZERO;
                td.run_slow = false;
                world.insert_resource(LocalPlayers::default());
                world.insert_resource(RollbackFrameCount(0));
                world.insert_resource(ConfirmedFrameCount(-1));
                world.insert_resource(MaxPredictionWindow(8));
                check(unsafe { sys::bgr_reset_session(engine(world)) });
            }
        }
    }
    world.insert_resource(td);
}

/// `handle_requests` (schedule_systems.rs:170-289).  The component half of every request — snapshots, checksums, the
/// compiled GgrsSchedule systems — is ONE engine call for the whole vector; the host half (resources, Time<GgrsTime>,
/// CPU-only systems) still runs bevy_ggrs' schedules request by request, and its `Checksum` (the XOR of the host-side
/// ChecksumParts, checksum.rs:88-99) is XORed into the engine's value for the same frame.
pub fn handle_requests<C: Config<Input = u8>>(requests: Vec<GgrsRequest<C>>, info: sys::bgr_session_info, world: &mut World) {
    let _span = bevy::log::tracing::info_span!("ggrs", name = "HandleRequests").entered();
    let mut cells = Vec::new();
    let mut host_parts: Vec<u128> = Vec::new();
    let mut reqs: Vec<sys::bgr_request> = Vec::with_capacity(requests.len());
    for r in requests {
        match r {
            GgrsRequest::SaveGameState { cell, frame } => {
                let _s = bevy::log::tracing::info_span!("ggrs", name = "SaveWorld").entered();
                world.run_schedule(SaveWorld);                                  // host-side resources + their ChecksumParts
                host_parts.push(world.resource::<Checksum>().0);
                cells.push(cell);
                reqs.push(sys::bgr_request { kind: sys::BGR_REQ_SAVE, frame, ..Default::default() });
            }
            GgrsRequest::LoadGameState { frame, .. } => {
                let _s = bevy::log::tracing::info_span!("ggrs", name = "LoadWorld").entered();
                world.insert_resource(RollbackFrameCount(frame));
                world.run_schedule(LoadWorld);
                reqs.push(sys::bgr_request { kind: sys::BGR_REQ_LOAD, frame, ..Default::default() });
            }
            GgrsRequest::AdvanceFrame { inputs } => {
                let _s = bevy::log::tracing::info_span!("ggrs", name = "AdvanceWorld").entered();
                let mut q = sys::bgr_request { kind: sys::BGR_REQ_ADVANCE, n_players: inputs.len() as u32, ..Default::default() };
                for (i, (input, status)) in inputs.iter().enumerate().take(sys::BGR_MAX_PLAYERS) { q.inputs[i] = *input; q.status[i] = *status as u8; }
                reqs.push(q);
                let next = world.resource::<RollbackFrameCount>().0 + 1;
                world.insert_resource(RollbackFrameCount(next));
                world.insert_resource(PlayerInputs::<C>(inputs));
                world.run_schedule(AdvanceWorld);                               // GgrsTime + whatever stayed on the CPU
                world.remove_resource::<PlayerInputs<C>>();
            }
        }
    }
    let e = engine(world);
    let mut out = [sys::bgr_checksum::default(); sys::BGR_MAX_REQUESTS];
    let mut n = 0u32;
    check(unsafe { sys::bgr_handle_requests(e, &info, reqs.as_ptr(), reqs.len() as u32, out.as_mut_ptr(), out.len() as u32, &mut n) });
    // cell.save(frame, None, checksum)  (schedule_systems.rs:231-236) — GGRS never receives state bytes
    for ((cell, cs), host) in cells.into_iter().zip(&out[..n as usize]).zip(host_parts) {
        cell.save(cs.frame, None, Some((((cs.hi as u128) << 64) | cs.lo as u128) ^ host));
    }
    let (mut frame, mut confirmed, mut maxp) = (0i32, 0i32, 0u32);
    unsafe { sys::bgr_rollback_frame_count(e, &mut frame); sys::bgr_confirmed_frame_count(e, &mut confirmed); sys::bgr_max_prediction_window(e, &mut maxp); }
    world.insert_resource(RollbackFrameCount(frame));
    world.insert_resource(ConfirmedFrameCount(confirmed));
    world.insert_resource(MaxPredictionWindow(maxp as usize));
}

/// A GgrsSchedule system of the game's own, written as CUDA source and compiled into the registration's kernel
/// (`bgr_add_user_system`; the contract is in include/bevy_ggrs_b200.h):
/// `BGR_SYSTEM_FN void NAME(const bgr_sys_ctx&, bgr_commands&, A&, const B&, ...)`, one parameter per bound column.
pub struct CudaSystem<'a> {
    pub name: &'a str,
    pub source: &'a str,
    pub columns: &'a [TypeId],
    pub params: &'a [u32],
}

/// The GgrsSchedule systems that run on the GPU, in schedule order, each with the component types it binds.
pub trait AddGpuSystems {
    fn add_gpu_systems(&mut self, systems: &[(GpuSystem, &[TypeId])]) -> &mut Self;
    fn add_cuda_system(&mut self, system: CudaSystem) -> &mut Self;
}
impl AddGpuSystems for App {
    fn add_gpu_systems(&mut self, systems: &[(GpuSystem, &[TypeId])]) -> &mut Self {
        for (s, cols) in systems {
            let ids: Vec<u32> = cols.iter().map(|t| self.world().resource::<Columns>().by_type[t]).collect();
            check(unsafe { sys::bgr_add_system(engine(self.world()), *s as u32, ids.as_ptr(), ids.len() as u32, core::ptr::null(), 0) });
        }
        self
    }
    fn add_cuda_system(&mut self, system: CudaSystem) -> &mut Self {
        let ids: Vec<u32> = system.columns.iter().map(|t| self.world().resource::<Columns>().by_type[t]).collect();
        let name = CString::new(system.name).expect("system name without NUL");
        let source = CString::new(system.source).expect("system source without NUL");
        check(unsafe {
            sys::bgr_add_user_system(engine(self.world()), name.as_ptr(), source.as_ptr(), ids.as_ptr(), ids.len() as u32,
                                     system.params.as_ptr(), system.params.len() as u32)
        });
        self
    }
}
