//! Raw declarations of `include/bevy_ggrs_b200.h` (ABI version 1).  One item per C declaration, same order.
//! SOURCE ONLY — never compiled in the build image (no Rust toolchain there).
#![allow(non_camel_case_types)]
use core::ffi::{c_char, c_int, c_void};

pub const BGR_ABI_VERSION: u32 = 1;
pub const BGR_MAX_PLAYERS: usize = 8;
pub const BGR_MAX_REQUESTS: usize = 80;
pub const BGR_MAX_CHECKSUM_COLUMNS: usize = 6;

pub const BGR_OK: c_int = 0;
pub const BGR_ERR_NO_SNAPSHOT: c_int = 4;
pub const BGR_ERR_NON_FINITE: c_int = 6;

pub const BGR_STRATEGY_COPY: u32 = 0;
pub const BGR_STRATEGY_CLONE: u32 = 1;
pub const BGR_STRATEGY_OPTIONAL: u32 = 0x100;
pub const BGR_MAX_OPTIONAL_COLUMNS: u32 = 7;
pub const BGR_HASH_BYTES: u32 = 1;
pub const BGR_HASH_FLAG_ASSERT_FINITE_F32: u32 = 1;

pub const BGR_SYS_PARTICLES_UPDATE: u32 = 1;
pub const BGR_SYS_PARTICLES_DESPAWN: u32 = 2;
pub const BGR_SYS_BOX_MOVE: u32 = 3;
pub const BGR_SYS_U32_ADD: u32 = 4;
pub const BGR_SYS_U32_SATSUB_DESPAWN: u32 = 5;
pub const BGR_SYS_U32_STORE_CALL_COUNT: u32 = 6;
pub const BGR_SYS_PARTICLES_SPAWN: u32 = 7;
pub const BGR_SYS_DESPAWN_ON_INPUT: u32 = 8;

pub const BGR_REQ_SAVE: u32 = 0;
pub const BGR_REQ_LOAD: u32 = 1;
pub const BGR_REQ_ADVANCE: u32 = 2;
pub const BGR_SESSION_NONE: u32 = 0;
pub const BGR_SESSION_SYNCTEST: u32 = 1;
pub const BGR_SESSION_P2P: u32 = 2;
pub const BGR_SESSION_SPECTATOR: u32 = 3;

pub const BGR_CFG_FORCE_STEPWISE: u32 = 1;
pub const BGR_CFG_SHARDED: u32 = 2;
pub const BGR_CFG_SKIP_UNCHANGED_PLANES: u32 = 4;

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct bgr_request {
    pub kind: u32,
    pub frame: i32,
    pub n_players: u32,
    pub inputs: [u8; BGR_MAX_PLAYERS],
    pub status: [u8; BGR_MAX_PLAYERS],
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct bgr_session_info {
    pub kind: u32,
    pub max_prediction: u32,
    pub check_distance: u32,
    pub confirmed_frame: i32,
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct bgr_checksum {
    pub frame: i32,
    pub has_checksum: u32,
    pub lo: u64,
    pub hi: u64,
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct bgr_partial {
    pub frame: i32,
    pub n_columns: u32,
    pub active: u64,
    pub total: u64,
    pub xor_: [u64; BGR_MAX_CHECKSUM_COLUMNS],
}

#[repr(C)]
pub struct bgr_config {
    pub abi_version: u32,
    pub device: i32,
    pub max_entities: u32,
    pub max_depth: u32,
    pub fps: u32,
    pub flags: u32,
    pub order_base: u64,
    pub stream: *mut c_void,
}

pub enum bgr_engine {}
#[allow(non_camel_case_types)]
pub enum bgr_group {}

extern "C" {
    pub fn bgr_abi_version() -> u32;
    pub fn bgr_last_error() -> *const c_char;
    pub fn bgr_engine_create(cfg: *const bgr_config, out: *mut *mut bgr_engine) -> c_int;
    pub fn bgr_engine_destroy(e: *mut bgr_engine);
    pub fn bgr_rollback_component(e: *mut bgr_engine, type_name: *const c_char, elem_bytes: u32, strategy: u32, column_out: *mut u32) -> c_int;
    pub fn bgr_checksum_component(e: *mut bgr_engine, column: u32, hash_kind: u32, byte_offset: u32, byte_len: u32, flags: u32) -> c_int;
    pub fn bgr_add_system(e: *mut bgr_engine, system: u32, columns: *const u32, n_columns: u32, params: *const u32, n_params: u32) -> c_int;
    pub fn bgr_add_user_system(e: *mut bgr_engine, name: *const c_char, cuda_source: *const c_char, columns: *const u32, n_columns: u32,
                               params: *const u32, n_params: u32) -> c_int;
    pub fn bgr_build(e: *mut bgr_engine) -> c_int;
    pub fn bgr_run_startup_system(e: *mut bgr_engine, system: u32) -> c_int;
    pub fn bgr_spawn(e: *mut bgr_engine, count: u32, first_row_out: *mut u32) -> c_int;
    pub fn bgr_despawn(e: *mut bgr_engine, row: u32) -> c_int;
    pub fn bgr_row_count(e: *mut bgr_engine, rows_out: *mut u32) -> c_int;
    pub fn bgr_active_count(e: *mut bgr_engine, active_out: *mut u64) -> c_int;
    pub fn bgr_write_component(e: *mut bgr_engine, column: u32, first_row: u32, count: u32, host_src: *const c_void, stride: u32) -> c_int;
    pub fn bgr_read_component(e: *mut bgr_engine, column: u32, first_row: u32, count: u32, host_dst: *mut c_void, stride: u32) -> c_int;
    pub fn bgr_read_alive(e: *mut bgr_engine, first_row: u32, count: u32, host_dst: *mut u8) -> c_int;
    pub fn bgr_remove_component(e: *mut bgr_engine, column: u32, row: u32) -> c_int;
    pub fn bgr_insert_component(e: *mut bgr_engine, column: u32, row: u32, value: *const c_void) -> c_int;
    pub fn bgr_has_component(e: *mut bgr_engine, column: u32, first_row: u32, count: u32, host_dst: *mut u8) -> c_int;
    pub fn bgr_host_alloc(bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn bgr_host_free(p: *mut c_void) -> c_int;
    pub fn bgr_download_begin(e: *mut bgr_engine, column: u32, byte_offset: u32, byte_len: u32, first_row: u32, count: u32, host_dst: *mut c_void, ticket_out: *mut u32) -> c_int;
    pub fn bgr_download_wait(e: *mut bgr_engine, ticket: u32) -> c_int;
    pub fn bgr_rollback_frame_count(e: *mut bgr_engine, out: *mut i32) -> c_int;
    pub fn bgr_set_rollback_frame_count(e: *mut bgr_engine, frame: i32) -> c_int;
    pub fn bgr_confirmed_frame_count(e: *mut bgr_engine, out: *mut i32) -> c_int;
    pub fn bgr_max_prediction_window(e: *mut bgr_engine, out: *mut u32) -> c_int;
    pub fn bgr_set_depth(e: *mut bgr_engine, depth: u32) -> c_int;
    pub fn bgr_confirm(e: *mut bgr_engine, confirmed_frame: i32) -> c_int;
    pub fn bgr_snapshot_frames(e: *mut bgr_engine, frames_out: *mut i32, cap: u32, n_out: *mut u32) -> c_int;
    pub fn bgr_peek(e: *mut bgr_engine, frame: i32, column: u32, first_row: u32, count: u32, host_dst: *mut c_void, stride: u32, alive_dst: *mut u8, found: *mut i32) -> c_int;
    pub fn bgr_save_world(e: *mut bgr_engine, checksum_out: *mut bgr_checksum) -> c_int;
    pub fn bgr_load_world(e: *mut bgr_engine) -> c_int;
    pub fn bgr_advance_world(e: *mut bgr_engine, inputs: *const u8, status: *const u8, n_players: u32) -> c_int;
    pub fn bgr_handle_requests(e: *mut bgr_engine, session: *const bgr_session_info, requests: *const bgr_request, n_requests: u32, checksums_out: *mut bgr_checksum, checksums_cap: u32, n_checksums_out: *mut u32) -> c_int;
    pub fn bgr_submit_requests(e: *mut bgr_engine, session: *const bgr_session_info, requests: *const bgr_request, n_requests: u32) -> c_int;
    pub fn bgr_collect(e: *mut bgr_engine, checksums_out: *mut bgr_checksum, checksums_cap: u32, n_checksums_out: *mut u32) -> c_int;
    pub fn bgr_last_partials(e: *mut bgr_engine, out: *mut bgr_partial, cap: u32, n_out: *mut u32) -> c_int;
    pub fn bgr_fold_partials(combined: *const bgr_partial, out: *mut bgr_checksum) -> c_int;
    pub fn bgr_collect_partials(e: *mut bgr_engine, partials_out: *mut bgr_partial, cap: u32, n_out: *mut u32) -> c_int;
    pub fn bgr_fold_partials_n(combined: *const bgr_partial, n: u32, out: *mut bgr_checksum) -> c_int;
    pub fn bgr_seahash(bytes: *const c_void, len: u64) -> u64;
    pub fn bgr_ggrs_time_delta_bits(fps: u32, frame: i32) -> u32;
    pub fn bgr_particle_rng_stream(seed: u64, state4_or_null: *const u64, n: u32, next_u64_out: *mut u64, range_out: *mut f32, low: f32, high: f32) -> c_int;
    pub fn bgr_splitmix64_stream(seed: u64, n: u32, out: *mut u64) -> c_int;
    pub fn bgr_launch_count(e: *mut bgr_engine, kernels_launched_out: *mut u64) -> c_int;
    pub fn bgr_slot_bytes(e: *mut bgr_engine, bytes_out: *mut u64) -> c_int;
    pub fn bgr_last_path(e: *mut bgr_engine, fused_out: *mut u32) -> c_int;
    pub fn bgr_generic_specialised(e: *mut bgr_engine, specialised_out: *mut u32) -> c_int;
    pub fn bgr_synchronize(e: *mut bgr_engine) -> c_int;
    pub fn bgr_stream(e: *mut bgr_engine, stream_out: *mut *mut c_void) -> c_int;
    pub fn bgr_trace_enable(e: *mut bgr_engine, capacity: u32) -> c_int;
    pub fn bgr_trace_read(e: *mut bgr_engine, rows_out: *mut u64, cap_launches: u32, n_out: *mut u32) -> c_int;
    pub fn bgr_host_profile(e: *mut bgr_engine, out: *mut u64, cap: u32) -> c_int;
    pub fn bgr_reset_session(e: *mut bgr_engine) -> c_int;
    pub fn bgr_shard_group_join(e: *mut bgr_engine, name: *const c_char, rank: u32, world_size: u32, timeout_ms: u32) -> c_int;
    pub fn bgr_shard_group_leave(e: *mut bgr_engine) -> c_int;
    pub fn bgr_group_join(name: *const c_char, rank: u32, world_size: u32, n_columns: u32, timeout_ms: u32) -> *mut bgr_group;
    pub fn bgr_group_leave(g: *mut bgr_group);
    pub fn bgr_group_publish(g: *mut bgr_group, group_seq: u64, partials: *const bgr_partial, n: u32) -> c_int;
    pub fn bgr_group_collect(g: *mut bgr_group, group_seq: u64, out: *mut bgr_checksum, cap: u32, n_out: *mut u32) -> c_int;
}
