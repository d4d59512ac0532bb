/*
 * bevy_ggrs_b200 — C ABI of the B200-native rollback snapshot / checksum / re-simulation engine.
 *
 * This is the drop-in boundary for ONE hot path of gschup/bevy_ggrs (reference paths are
 * relative to the upstream repo, v0.20.0):
 *
 *   - per-tick save/load of the registered component columns       src/snapshot/component_snapshot.rs:66-123
 *   - the newest-first ring of frame snapshots                      src/snapshot/mod.rs:94-271
 *   - the per-frame desync checksum                                 src/snapshot/{checksum,component_checksum,entity_checksum}.rs
 *   - the request loop that replays N frames after a rollback       src/schedule_systems.rs:170-289 (handle_requests)
 *   - the registered stress-test systems of GgrsSchedule            examples/stress_tests/particles.rs:272-289
 *
 * Everything lives in HBM: registered columns are stored word-planar (one plane of 4-byte
 * words per field word, see DESIGN.md "Data layout"), snapshots are a ring of frame slots
 * with the same layout, and a whole Vec<GgrsRequest> ( Load + N x (Advance, Save) + ... )
 * is executed by ONE kernel launch.  GGRS never receives state bytes
 * (`cell.save(frame, None, checksum)`, schedule_systems.rs:235-236), so the only things that
 * cross this boundary per tick are the request list (in) and one u128 checksum per Save (out).
 *
 * Conventions
 *   - plain C, fixed-width ints, no torch / CUDA types in signatures (a cudaStream_t is
 *     passed as void*).
 *   - every call returns a bgr_status; on failure bgr_last_error() holds the text of the
 *     panic the reference would have raised (e.g. "Could not rollback to 99: no snapshot at
 *     that moment could be found.", mod.rs:209-212).  A Rust shim turns non-zero into panic!.
 *   - one caller thread at a time per engine (the reference calls from an exclusive system,
 *     schedule_systems.rs:19,170).
 *   - u128 checksums cross as two u64 (lo, hi); hi is always 0 in the reference because every
 *     part is `u64 as u128` (component_checksum.rs:95, entity_checksum.rs:43).
 *   - the library FAILS LOUDLY (BGR_ERR_CUDA) when no sm_100 device is usable; there is no
 *     CPU fallback anywhere behind this header.
 */
#ifndef BEVY_GGRS_B200_H
#define BEVY_GGRS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BGR_API __attribute__((visibility("default")))

#define BGR_ABI_VERSION 1u
#define BGR_MAX_PLAYERS 8u      /* every handle 0..7 reaches the systems (PlayerInputs<T>.0[handle], box_game.rs:171) */
#define BGR_MAX_REQUESTS 80u  /* max requests per bgr_handle_requests call (2*32+2 for a 32-frame SyncTest) */

typedef enum bgr_status {
    BGR_OK = 0,
    BGR_ERR_INVALID_ARGUMENT = 1,
    BGR_ERR_STATE = 2,            /* call order violated (e.g. register after build) */
    BGR_ERR_CUDA = 3,             /* no usable GPU / CUDA runtime failure — never falls back to CPU */
    BGR_ERR_NO_SNAPSHOT = 4,      /* GgrsSnapshots::rollback / get panic, mod.rs:207-230 */
    BGR_ERR_MISSING_RESOURCE = 5, /* `expect(...)` on RollbackFrameCount / LocalInputs, schedule_systems.rs:90-92,245-246 */
    BGR_ERR_NON_FINITE = 6,       /* assert!(is_finite) in the stress hashers, particles.rs:111-114,212-215 */
    BGR_ERR_CAPACITY = 7,         /* more rows / slots / requests than configured */
    BGR_ERR_UNSUPPORTED = 8
} bgr_status;

/* Strategy<T> (src/snapshot/strategy.rs:22-83).  Copy and Clone of a POD are both a bitwise
 * copy; ReflectStrategy is out of scope (boxed dynamic reflection, SURVEY.md §2 row 5). */
typedef enum bgr_strategy { BGR_STRATEGY_COPY = 0, BGR_STRATEGY_CLONE = 1 } bgr_strategy;
/* OR into `strategy`: single entities may lose / regain this component inside the rollback window
 * (`Option<&mut S::Target>` in ComponentSnapshotPlugin::load, src/snapshot/component_snapshot.rs:99-115).  Save stores
 * the component only for the entities that have it, Load updates / removes / inserts / leaves alone accordingly, the
 * checksum and the GgrsSchedule systems only see entities that have it.  At most BGR_MAX_OPTIONAL_COLUMNS columns. */
#define BGR_STRATEGY_OPTIONAL 0x100u
#define BGR_MAX_OPTIONAL_COLUMNS 7

/* How `checksum_component::<T>(hasher)` hashes one element (rollback_app.rs:227-232,
 * component_checksum.rs:44-48).  BGR_HASH_BYTES = seahash over elem[offset .. offset+len):
 * this is what `#[derive(Hash)]` produces for a POD of ints (fields appended little-endian)
 * and what the particles hashers do with `x.to_bits()` (particles.rs:107-120, 207-222). */
typedef enum bgr_hash_kind { BGR_HASH_NONE = 0, BGR_HASH_BYTES = 1 } bgr_hash_kind;
#define BGR_HASH_FLAG_ASSERT_FINITE_F32 1u /* every 4-byte word in the range must be a finite f32 */

/* Systems that can be added to GgrsSchedule (`add_systems(GgrsSchedule, ...)`, lib.rs:73-74).
 * These are compiled in; a game's own systems are added as CUDA source with bgr_add_user_system below. */
typedef enum bgr_system {
    /* update_particles, particles.rs:272-280.  cols = {Transform(40B), Velocity(12B)} */
    BGR_SYS_PARTICLES_UPDATE = 1,
    /* despawn_particles, particles.rs:282-289.  cols = {Ttl(8B)} */
    BGR_SYS_PARTICLES_DESPAWN = 2,
    /* move_cube_system, box_game.rs:154-206.  cols = {Transform(40B), Velocity(12B)}; player handle = row */
    BGR_SYS_BOX_MOVE = 3,
    /* `x.0 += k` on a u32 field (tests/component_rollback.rs:25-29 increment_score).
     * cols = {C}; params = {byte_offset, k} */
    BGR_SYS_U32_ADD = 4,
    /* `h = h.saturating_sub(k); if h == 0 { despawn }` (tests/synctest.rs:38-45 decrease_health).
     * cols = {C}; params = {byte_offset, k} */
    BGR_SYS_U32_SATSUB_DESPAWN = 5,
    /* writes a host-side call counter that is NOT rolled back into a u32 field — the
     * deliberately non-deterministic system of tests/synctest.rs:83-125.
     * cols = {C}; params = {byte_offset} */
    BGR_SYS_U32_STORE_CALL_COUNT = 6,
    /* spawn_particles.run_if(spawn_pressed), particles.rs:243-270: when any player's input has INPUT_SPAWN
     * (1 << 4) set, appends `rate` rows: Transform::default(), Velocity(random_range(-200..200) x2, 0), Ttl(ttl),
     * Rollback.  Draws from the ParticleRng resource (Xoshiro256PlusPlus::seed_from_u64(seed)), which the engine
     * keeps host-side and rolls back with every snapshot (rollback_resource_with_clone::<ParticleRng>, :200).
     * Commands are deferred: the new rows exist from the end of the frame on and are not updated in it.
     * cols = {Transform(40B), Velocity(12B), Ttl(8B)}; params = {rate, ttl, seed_lo, seed_hi} */
    BGR_SYS_PARTICLES_SPAWN = 7,
    /* `if inputs[player].0 == value { commands.entity(e).despawn() }` for every entity that has component C — the
     * shape of tests/hierarchy.rs:36-45 delete_child_system (there the child is reached through the parent's `Children`;
     * here C is the child's own `ChildOf`, an optional 8-byte column holding the parent's RollbackOrdered index: row
     * indices are stable across rollback, so the hierarchy needs neither ChildOfSnapshotPlugin's remapping
     * (childof_snapshot.rs) nor MapEntities (component_map.rs)).  cols = {C}; params = {player_handle, value} */
    BGR_SYS_DESPAWN_ON_INPUT = 8
} bgr_system;
#define BGR_INPUT_SPAWN 0x10u /* INPUT_SPAWN, particles.rs:75 */

/* GgrsRequest<T> (ggrs; consumed at schedule_systems.rs:222-269). Input type is u8
 * (particles.rs:73 `GgrsConfig<u8>`, box_game.rs:27-29 `BoxInput(u8)`). */
typedef enum bgr_request_kind { BGR_REQ_SAVE = 0, BGR_REQ_LOAD = 1, BGR_REQ_ADVANCE = 2 } bgr_request_kind;
typedef enum bgr_input_status { BGR_INPUT_CONFIRMED = 0, BGR_INPUT_PREDICTED = 1, BGR_INPUT_DISCONNECTED = 2 } bgr_input_status;

typedef struct bgr_request {
    uint32_t kind;                    /* bgr_request_kind */
    int32_t frame;                    /* SaveGameState{frame} / LoadGameState{frame}; ignored for Advance */
    uint32_t n_players;               /* AdvanceFrame{inputs}.len() */
    uint8_t inputs[BGR_MAX_PLAYERS];  /* PlayerInputs<T>.0[i].0 */
    uint8_t status[BGR_MAX_PLAYERS];  /* PlayerInputs<T>.0[i].1 (bgr_input_status) */
} bgr_request;

/* What handle_requests reads from the Session each request (schedule_systems.rs:195-220). */
typedef enum bgr_session_kind {
    BGR_SESSION_NONE = 0, BGR_SESSION_SYNCTEST = 1, BGR_SESSION_P2P = 2, BGR_SESSION_SPECTATOR = 3
} bgr_session_kind;

typedef struct bgr_session_info {
    uint32_t kind;            /* bgr_session_kind */
    uint32_t max_prediction;  /* s.max_prediction() (forced to 0 for spectators, :200) */
    uint32_t check_distance;  /* SyncTest: s.check_distance() (:207) */
    int32_t confirmed_frame;  /* P2P: s.confirmed_frame() (:205) */
} bgr_session_info;

/* `Checksum(u128)` (checksum.rs:49) handed to `cell.save(frame, None, checksum)`. */
typedef struct bgr_checksum {
    int32_t frame;
    uint32_t has_checksum;  /* always 1 (ChecksumPlugin is part of GgrsPlugin, lib.rs:257) */
    uint64_t lo, hi;
} bgr_checksum;

/* Raw per-Save partials of ONE shard, before the cross-shard fold (multi-GPU, SURVEY §8e):
 * xor[c] is the XOR over live rows of the per-entity hash of checksummed column c
 * (component_checksum.rs:81-90, before the final `result.hash()` at :93); active = live rows. */
#define BGR_MAX_CHECKSUM_COLUMNS 6u
typedef struct bgr_partial {
    int32_t frame;
    uint32_t n_columns;
    uint64_t active;      /* active_entities.iter().len() of this shard, entity_checksum.rs:38 */
    uint64_t total;       /* rollback_ordered.len() of this shard, entity_checksum.rs:41 */
    uint64_t xor_[BGR_MAX_CHECKSUM_COLUMNS];
} bgr_partial;

typedef struct bgr_config {
    uint32_t abi_version;   /* BGR_ABI_VERSION */
    int32_t device;         /* CUDA ordinal */
    uint32_t max_entities;  /* row capacity of this shard */
    uint32_t max_depth;     /* frame slots allocated in HBM; >= the largest MaxPredictionWindow used (+1 for SyncTest d == p-1 is not needed) */
    uint32_t fps;           /* RollbackFrameRate, time.rs:19-26 (default 60) */
    uint32_t flags;         /* BGR_CFG_* */
    uint64_t order_base;    /* RollbackOrdered index of local row 0 (entity-range sharding); 0 on one GPU */
    void* stream;           /* cudaStream_t to run on; NULL = engine creates its own */
} bgr_config;
#define BGR_CFG_FORCE_STEPWISE 1u  /* never use the fused one-launch program kernel (debug / A-B tests) */
#define BGR_CFG_SHARDED 2u         /* handle_requests returns partials only; caller folds across shards */
/* OPT-IN, off by default: do not rewrite word planes whose content is provably identical to what the target
 * image already holds.  The engine tracks a content version for the planes no registered system writes
 * (e.g. Transform.rotation/scale in the stress test): a Save into a slot that already holds the current version
 * skips those planes, and so does a Load.  Snapshots stay complete images (peek / load need no indirection) and
 * every observable result is unchanged; only redundant HBM stores are elided.  The reference clones every
 * registered component on every save (component_snapshot.rs:71-75), so the default keeps doing exactly that. */
#define BGR_CFG_SKIP_UNCHANGED_PLANES 4u

typedef struct bgr_engine bgr_engine;

/* ---- lifetime ------------------------------------------------------------------------ */
BGR_API uint32_t bgr_abi_version(void);
BGR_API const char* bgr_last_error(void);  /* thread-local text of the last failure */
BGR_API int bgr_engine_create(const bgr_config* cfg, bgr_engine** out);
BGR_API void bgr_engine_destroy(bgr_engine* e);

/* ---- registration  (RollbackApp, src/snapshot/rollback_app.rs:31-248) ------------------ */
/* rollback_component_with_copy::<T>() / rollback_component_with_clone::<T>() (:157-183) */
BGR_API int bgr_rollback_component(bgr_engine* e, const char* type_name, uint32_t elem_bytes,
                                   uint32_t strategy, uint32_t* column_out);
/* checksum_component::<T>(hasher) / checksum_component_with_hash::<T>() (:199-232) */
BGR_API int bgr_checksum_component(bgr_engine* e, uint32_t column, uint32_t hash_kind,
                                   uint32_t byte_offset, uint32_t byte_len, uint32_t flags);
/* add_systems(GgrsSchedule, system) — systems run in insertion order each AdvanceFrame */
BGR_API int bgr_add_system(bgr_engine* e, uint32_t system, const uint32_t* columns, uint32_t n_columns,
                           const uint32_t* params, uint32_t n_params);
/* add_systems(GgrsSchedule, NAME) for a system of the game's own, given as CUDA source and compiled into the
 * registration's own kernel at bgr_build (NVRTC).  It runs in add_systems order, interleaved with the compiled-in systems:
 *
 *     struct Velocity { float x, y, z; };
 *     BGR_SYSTEM_FN void apply_drag(const bgr_sys_ctx& ctx, bgr_commands& cmd, Velocity& v) {
 *         const float k = bgr_f32(ctx.params[0]);
 *         v.x = v.x * k; v.y = v.y * k; v.z = v.z * k;
 *         if (v.x == 0.0f && v.y == 0.0f) cmd.despawn();
 *     }
 *
 *   - signature: `BGR_SYSTEM_FN void NAME(const bgr_sys_ctx&, bgr_commands&, A&, const B&, ...)`, one parameter per bound
 *     column in binding order (1 to 4).  A..: the game's POD structs, declared in the same source, sizeof == the column's
 *     elem_bytes (a static_assert naming the column checks it).  `const T&` is `&T` and is never written back; `T&` is
 *     `&mut T`.  The same column may not be bound twice.
 *   - entities: every entity that exists and has every bound column (`Query<(&mut A, &B)>`, optional columns included).
 *     Every system of a frame sees entity presence as it was before the frame.  One entity at a time: no reads of others.
 *   - cmd.despawn() is deferred to after the last system of the frame, like every despawn command.
 *   - bgr_sys_ctx: dt (Time<GgrsTime> delta), frame (RollbackFrameCount inside AdvanceWorld, after its `+= 1`),
 *     n_players / inputs[8] (PlayerInputs<T>), order (the entity's RollbackOrdered index, order_base + row: the player
 *     handle of box_game-style systems), params[8] (`params`, constant in the generated kernel; bgr_f32 reads one as a
 *     float).  Input status is not exposed.
 *   - floating point: + - * / and sqrtf are bit-exact with a CPU build (-fmad=false; g++ -ffp-contract=off on the host);
 *     transcendentals (powf, sinf, ...) are not.
 *   - the source has no #include (the API, csrc/user_system.cuh, is already included), no __global__, no __shared__, no
 *     mutable __device__ globals.  It is compiled inside a namespace of its own (two systems may each declare a
 *     `struct Velocity`) behind `#line 1 "NAME"`, so compile errors point at the source's own lines.
 * Checked here: NAME is a C identifier not used by another user system, the source is at most 64 KB, the columns exist
 * and are distinct, n_params <= 8, at most 8 systems in total, and the call comes before bgr_build.  bgr_build then fails
 * with BGR_ERR_INVALID_ARGUMENT and NVRTC's log in bgr_last_error() when the source does not compile, and with
 * BGR_ERR_UNSUPPORTED when the generated kernel cannot be had: no NVRTC or kernel sources, BGR_TUNE_JIT=0 or
 * BGR_TUNE_GENERIC=0, BGR_CFG_FORCE_STEPWISE, BGR_SYS_PARTICLES_SPAWN in the same registration, or more than 24 words
 * (96 bytes) of registered columns per entity.  The engine stays destroyable after any of these failures. */
BGR_API int bgr_add_user_system(bgr_engine* e, const char* name, const char* cuda_source, const uint32_t* columns,
                                uint32_t n_columns, const uint32_t* params, uint32_t n_params);
/* end of App::build: allocates live columns + max_depth frame slots in HBM */
BGR_API int bgr_build(bgr_engine* e);
/* add_systems(Startup, system): run a registered GgrsSchedule system once, outside the rollback loop
 * (particles.rs:232 `add_systems(Startup, spawn_particles)` — the initial burst).  Only BGR_SYS_PARTICLES_SPAWN. */
BGR_API int bgr_run_startup_system(bgr_engine* e, uint32_t system);

/* ---- entity population (Rollback marker, src/snapshot/rollback.rs:23-94) ---------------- */
/* `commands.spawn((..., Rollback))` x count: appends rows, RollbackOrdered index = order_base + row */
BGR_API int bgr_spawn(bgr_engine* e, uint32_t count, uint32_t* first_row_out);
BGR_API int bgr_despawn(bgr_engine* e, uint32_t row);
BGR_API int bgr_row_count(bgr_engine* e, uint32_t* rows_out);   /* RollbackOrdered::len() */
BGR_API int bgr_active_count(bgr_engine* e, uint64_t* active_out);
/* ECS column <-> HBM planes.  host buffers are arrays of T with `stride` bytes between
 * elements (stride >= elem_bytes; stride = size_of::<T>() on the Rust side). */
BGR_API int bgr_write_component(bgr_engine* e, uint32_t column, uint32_t first_row, uint32_t count,
                                const void* host_src, uint32_t stride);
BGR_API int bgr_read_component(bgr_engine* e, uint32_t column, uint32_t first_row, uint32_t count,
                               void* host_dst, uint32_t stride);
BGR_API int bgr_read_alive(bgr_engine* e, uint32_t first_row, uint32_t count, uint8_t* host_dst);

/* ---- per-entity component presence (columns registered with BGR_STRATEGY_OPTIONAL) ----------
 * bgr_remove_component = `commands.entity(e).remove::<T>()`, bgr_insert_component = `.insert(value)` applied to the live
 * world between request vectors (value: elem_bytes bytes); bgr_has_component writes 1 per row that is alive and has it. */
BGR_API int bgr_remove_component(bgr_engine* e, uint32_t column, uint32_t row);
BGR_API int bgr_insert_component(bgr_engine* e, uint32_t column, uint32_t row, const void* value);
BGR_API int bgr_has_component(bgr_engine* e, uint32_t column, uint32_t first_row, uint32_t count, uint8_t* host_dst);

/* ---- asynchronous mirror download: what the ECS side reads back every tick -----------------
 * In the reference the world lives in host memory and everything after GgrsSchedule (rendering via Transform,
 * examples/stress_tests/particles.rs:191-196; game logic outside the rollback schedule) reads it there.  With the
 * world in HBM the shim mirrors only the fields those readers need: bytes [byte_offset, byte_offset+byte_len) of
 * every element of `column` for rows [first_row, first_row+count), packed densely (byte_len bytes per row) into
 * `host_dst`.  byte_offset and byte_len must be multiples of 4.
 *
 * bgr_download_begin is ordered after every request vector submitted so far (it sees the live world those leave
 * behind), returns without waiting for the GPU, and does not delay later submits: the fields are packed into a device
 * staging buffer on the engine's stream and cross PCIe on a separate copy stream.  `host_dst` should come from
 * bgr_host_alloc (page-locked); it must not be read before bgr_download_wait(ticket) returns.  At most
 * BGR_MAX_DOWNLOADS may be in flight. */
#define BGR_MAX_DOWNLOADS 4
BGR_API int bgr_host_alloc(size_t bytes, void** out);
BGR_API int bgr_host_free(void* p);
BGR_API int bgr_download_begin(bgr_engine* e, uint32_t column, uint32_t byte_offset, uint32_t byte_len,
                               uint32_t first_row, uint32_t count, void* host_dst, uint32_t* ticket_out);
BGR_API int bgr_download_wait(bgr_engine* e, uint32_t ticket);

/* ---- frame resources (src/snapshot/mod.rs:66-77, lib.rs:116-117) ------------------------ */
BGR_API int bgr_rollback_frame_count(bgr_engine* e, int32_t* out);
BGR_API int bgr_set_rollback_frame_count(bgr_engine* e, int32_t frame);
BGR_API int bgr_confirmed_frame_count(bgr_engine* e, int32_t* out);
BGR_API int bgr_max_prediction_window(bgr_engine* e, uint32_t* out);
/* the session-less branch of run_ggrs_schedules (schedule_systems.rs:70-79): RollbackFrameCount(0),
 * ConfirmedFrameCount(-1), MaxPredictionWindow(8) */
BGR_API int bgr_reset_session(bgr_engine* e);

/* ---- snapshot ring (GgrsSnapshots, src/snapshot/mod.rs:94-271) -------------------------- */
BGR_API int bgr_set_depth(bgr_engine* e, uint32_t depth);                 /* :120-135 */
BGR_API int bgr_confirm(bgr_engine* e, int32_t confirmed_frame);          /* :182-199 */
BGR_API int bgr_snapshot_frames(bgr_engine* e, int32_t* frames_out, uint32_t cap, uint32_t* n_out); /* newest first */
/* peek(frame) (:233-240): *found = 0 if no snapshot for `frame`; otherwise copies the rows. */
BGR_API int bgr_peek(bgr_engine* e, int32_t frame, uint32_t column, uint32_t first_row, uint32_t count,
                     void* host_dst, uint32_t stride, uint8_t* alive_dst, int32_t* found);

/* ---- the three schedules, one at a time (SnapshotPlugin-only users: benches/bench.rs:18-27,
 *      mod.rs:510-535 save_world / advance_frame / load_world helpers) -------------------- */
BGR_API int bgr_save_world(bgr_engine* e, bgr_checksum* checksum_out);         /* world.run_schedule(SaveWorld) */
BGR_API int bgr_load_world(bgr_engine* e);                                     /* world.run_schedule(LoadWorld) at RollbackFrameCount */
BGR_API int bgr_advance_world(bgr_engine* e, const uint8_t* inputs, const uint8_t* status,
                              uint32_t n_players);                             /* world.run_schedule(AdvanceWorld); caller bumps the frame count */

/* ---- THE HOT LOOP: handle_requests (src/schedule_systems.rs:170-289) ------------------- */
/* Executes the whole request vector; one fused kernel launch when the registered systems
 * match a compiled bundle, otherwise one launch per request.  Writes one bgr_checksum per
 * SaveGameState, in request order, host-visible on return. */
BGR_API int bgr_handle_requests(bgr_engine* e, const bgr_session_info* session,
                                const bgr_request* requests, uint32_t n_requests,
                                bgr_checksum* checksums_out, uint32_t checksums_cap, uint32_t* n_checksums_out);
/* Asynchronous pair: submit enqueues on the engine stream and returns; collect waits and
 * returns the checksums of the oldest un-collected submit.  At most 8 submits may be un-collected.
 * Entry points that read or edit the world (bgr_read_component, bgr_spawn, bgr_peek ...) wait for the submitted
 * vectors but leave their results queued for bgr_collect; bgr_handle_requests (and the one-schedule helpers above)
 * return BGR_ERR_STATE while submits are un-collected. */
BGR_API int bgr_submit_requests(bgr_engine* e, const bgr_session_info* session,
                                const bgr_request* requests, uint32_t n_requests);
BGR_API int bgr_collect(bgr_engine* e, bgr_checksum* checksums_out, uint32_t checksums_cap,
                        uint32_t* n_checksums_out);
/* Sharded engines (BGR_CFG_SHARDED): raw partials of the last collected call, and the fold
 * that turns cross-shard combined partials into the frame checksum
 * (component_checksum.rs:93-95, entity_checksum.rs:35-43, checksum.rs:88-99). */
BGR_API int bgr_last_partials(bgr_engine* e, bgr_partial* out, uint32_t cap, uint32_t* n_out);
BGR_API int bgr_fold_partials(const bgr_partial* combined, bgr_checksum* out);
/* bgr_collect that writes the raw partials of the collected call straight into caller memory (sharded hot loop:
 * no per-tick allocation), and the fold over an array of already combined partials. */
BGR_API int bgr_collect_partials(bgr_engine* e, bgr_partial* partials_out, uint32_t cap, uint32_t* n_out);
BGR_API int bgr_fold_partials_n(const bgr_partial* combined, uint32_t n, bgr_checksum* out);

/* ---- shard group: the cross-shard step inside the engine (multi-GPU, one process per GPU, one node) -----------------
 * Entity-range shards never exchange state (SURVEY.md §8e: systems read no other entity, box_game.rs:162-169; the
 * checksum is an XOR over entities, component_checksum.rs:88-89).  The only exchange is 64 bytes of partials per
 * SaveGameState.  After every rank's BGR_CFG_SHARDED engine has joined the same group, bgr_handle_requests /
 * bgr_collect on ANY rank return the frame checksum of the WHOLE world (has_checksum = 1) — what
 * `cell.save(frame, None, checksum)` needs (schedule_systems.rs:231-236) — with no call outside this library:
 * the result blocks live in one shared host segment that every rank's GPU stores into and every rank's CPU polls.
 * Every rank must be handed the same request vectors in the same order (they all replay the same GGRS session).
 * `name` must be unique per group instance (e.g. "<launcher pid>_<port>"); timeout_ms = 0 selects 60 s. */
BGR_API int bgr_shard_group_join(bgr_engine* e, const char* name, uint32_t rank, uint32_t world_size, uint32_t timeout_ms);
BGR_API int bgr_shard_group_leave(bgr_engine* e);
/* the group's host logic without an engine (no GPU call): CPU tests publish partials computed elsewhere */
typedef struct bgr_group bgr_group;
BGR_API bgr_group* bgr_group_join(const char* name, uint32_t rank, uint32_t world_size, uint32_t n_columns, uint32_t timeout_ms);
BGR_API void bgr_group_leave(bgr_group* g);
BGR_API int bgr_group_publish(bgr_group* g, uint64_t group_seq, const bgr_partial* partials, uint32_t n);  /* group_seq = 1, 2, ... */
BGR_API int bgr_group_collect(bgr_group* g, uint64_t group_seq, bgr_checksum* out, uint32_t cap, uint32_t* n_out);

/* ---- checksum_hasher() (src/snapshot/mod.rs:315-317) for host-side parts -------------------------------
 * Resources stay on the host (a few bytes, not data-parallel).  A shim that registers
 * `checksum_resource_with_hash::<R>()` (resource_checksum.rs:63-82) computes `part = bgr_seahash(bytes of R)`
 * per Save and XORs it into the engine's checksum (ChecksumPlugin::update, checksum.rs:88-99). */
BGR_API uint64_t bgr_seahash(const void* bytes, uint64_t len);

/* ---- ParticleRng arithmetic on its own (host only; examples/stress_tests/particles.rs:125-128, 258-270) -------
 * The Xoshiro256PlusPlus stream spawn_particles draws from: `state4_or_null` = Xoshiro256PlusPlus::from_seed state
 * words, or NULL for seed_from_u64(seed).  next_u64_out[i] = the i-th next_u64(); range_out[i] = the i-th
 * random_range(low..high) of an identical, separate generator.  bgr_splitmix64_stream = rand_xoshiro's SplitMix64.
 * Exposed so that published known-answer vectors run against the product's own code. */
BGR_API int bgr_particle_rng_stream(uint64_t seed, const uint64_t* state4_or_null, uint32_t n, uint64_t* next_u64_out,
                                    float* range_out, float low, float high);
BGR_API int bgr_splitmix64_stream(uint64_t seed, uint32_t n, uint64_t* out);

/* ---- GgrsTime (src/time.rs:63-76): delta_secs of the step that ends at `frame` ---------- */
BGR_API uint32_t bgr_ggrs_time_delta_bits(uint32_t fps, int32_t frame);

/* ---- introspection for benches / tests --------------------------------------------------- */
BGR_API int bgr_launch_count(bgr_engine* e, uint64_t* kernels_launched_out);
BGR_API int bgr_slot_bytes(bgr_engine* e, uint64_t* bytes_out);  /* algorithmic bytes of one frame slot at the current row count */
BGR_API int bgr_last_path(bgr_engine* e, uint32_t* fused_out);   /* 1 if the last handle_requests used the fused program kernel */
/* 1 if bgr_build compiled this registration's own kernel (NVRTC specialisation of the generic one-launch program,
 * csrc/generic_program_jit.cuh): every non-bundle request vector then runs on it; 0 = the interpreter kernel (same results).
 * Env BGR_TUNE_JIT: 0 never, 1 (default) engines created for >= 16384 entities or with user systems, 2 always. */
BGR_API int bgr_generic_specialised(bgr_engine* e, uint32_t* specialised_out);
BGR_API int bgr_synchronize(bgr_engine* e);
BGR_API int bgr_stream(bgr_engine* e, void** stream_out);        /* the cudaStream_t the engine launches on (timing events) */
/* device-side launch trace: 4 x u64 per fused launch after the call, up to `capacity` launches (GPU globaltimer ns):
 * [0] first block started, [1] last block finished its tiles, [2] results + completion word written, [3] reserved.
 * bgr_trace_read copies the rows out (waits for the GPU).  capacity 0 disables. */
BGR_API int bgr_trace_enable(bgr_engine* e, uint32_t capacity);
BGR_API int bgr_trace_read(bgr_engine* e, uint64_t* rows_out, uint32_t cap_launches, uint32_t* n_out);
/* cumulative host-side time of the hot loop: out[0] request vectors, [1] ns compiling requests, [2] ns enqueueing the
 * launch, [3] ns waiting for the completion word, [4] ns folding results (cap <= 8) */
BGR_API int bgr_host_profile(bgr_engine* e, uint64_t* out, uint32_t cap);

/* ---- host-side ring bookkeeping on its own ------------------------------------------------------
 * The frame -> HBM-slot queue the engine keeps for GgrsSnapshots (mod.rs:94-271), exposed without
 * an engine so the reference's 11 ring unit tests (mod.rs:365-508) run against it on a CPU-only
 * box.  Pure host logic, no GPU call. */
typedef struct bgr_ring bgr_ring;
BGR_API bgr_ring* bgr_ring_create(uint32_t n_slots);
BGR_API void bgr_ring_destroy(bgr_ring* r);
BGR_API uint32_t bgr_ring_depth(bgr_ring* r);
BGR_API int bgr_ring_set_depth(bgr_ring* r, uint32_t depth);
BGR_API int bgr_ring_push(bgr_ring* r, int32_t frame, uint32_t* slot_out);
BGR_API int bgr_ring_confirm(bgr_ring* r, int32_t frame);
BGR_API int bgr_ring_rollback(bgr_ring* r, int32_t frame, uint32_t* slot_out);
BGR_API int bgr_ring_get(bgr_ring* r, uint32_t* slot_out);
BGR_API int bgr_ring_peek(bgr_ring* r, int32_t frame, uint32_t* slot_out, int32_t* found);

#ifdef __cplusplus
}
#endif
#endif /* BEVY_GGRS_B200_H */
