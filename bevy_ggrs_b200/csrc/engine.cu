// bevy_ggrs_b200 engine: host logic of the rollback hot path + the C ABI of include/bevy_ggrs_b200.h.
//
// Host side restates, request by request, what handle_requests does to the frame resources
// (reference src/schedule_systems.rs:189-270) and to the snapshot ring (src/snapshot/mod.rs:144-270),
// compiles the whole request vector into a small op program, and launches ONE fused kernel
// (kernels.cuh: k_particles_program) — or, for schemas/systems without a compiled bundle, one
// generic kernel per request ("stepwise" path).  No CPU compute path exists: without a GPU every
// entry point that touches state returns BGR_ERR_CUDA.
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>  // header-only; a no-op unless a profiler is attached

#include <algorithm>
#include <array>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <string>
#include <vector>

#include "../../include/bevy_ggrs_b200.h"
#include "kernels.cuh"
#include "particle_rng.hpp"
#include "ring.hpp"
#include "seahash.cuh"
#include "shard_group.hpp"
#include "tma_copy.cuh"
#include "generic_program.cuh"
#include "jit.hpp"

using namespace bgr;

namespace {

thread_local std::string g_err;
int fail(int status, const std::string& text) { g_err = text; return status; }

#define CUDA_TRY(expr)                                                                              \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess)                                                                      \
            return fail(BGR_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));          \
    } while (0)

struct Column {
    std::string name;
    uint32_t elem_bytes = 0, words = 0, first_plane = 0, strategy = 0;
    uint32_t hash_kind = BGR_HASH_NONE, hash_off = 0, hash_len = 0, hash_flags = 0;
    int ck_slot = -1;  // index among checksummed columns (registration order)
    uint32_t absent = 0;  // optional column: its absent bit in the per-row mask byte (kernels.cuh row_matches)
};

// Internal id of a user system (bgr_add_user_system): never a bgr_system value.  It only runs on the registration's own
// kernel, where its SysSpec::param is its index among the user systems.
constexpr uint32_t kSysUser = 0x100;

struct SystemReg {
    uint32_t id = 0;
    std::vector<uint32_t> cols, params;
    std::string name, source;  // user systems: the function's name and its CUDA source
};

bool has_user_systems(const std::vector<SystemReg>& systems) {
    for (const SystemReg& sy : systems)
        if (sy.id == kSysUser) return true;
    return false;
}

constexpr uint32_t kReqAdvanceNoBump = 100;  // bgr_advance_world: caller already bumped RollbackFrameCount

constexpr uint32_t kMaxSpawnVals = 1u << 16;  // particles spawned by one request vector

// Every host-side resource handle_requests / the schedules mutate.  A request vector is compiled
// against a copy and committed only if the whole vector is valid.
struct HostState {  // trivially copyable: copying it per call must not allocate
    SlotRing ring;
    std::array<uint32_t, SlotRing::kMaxSlots> slot_rows{};        // RollbackOrdered::len() captured by each snapshot (mod.rs:339)
    std::array<uint64_t, SlotRing::kMaxSlots> slot_elapsed_ns{};  // Time<GgrsTime> captured by each snapshot (time.rs:100)
    int32_t frame_count = 0;                // RollbackFrameCount (mod.rs:66-67)
    int32_t confirmed = 0;                  // ConfirmedFrameCount (mod.rs:76-77), init_resource -> 0
    bool has_maxpred = false;               // MaxPredictionWindow inserted? (lib.rs:116-117)
    uint32_t maxpred = 0;
    uint64_t elapsed_ns = 0;                // Time<GgrsTime>::elapsed
    uint32_t n_rows = 0;                    // RollbackOrdered::len()
    uint32_t call_count = 0;                // un-rolled-back counter of BGR_SYS_U32_STORE_CALL_COUNT
    ParticleRng rng;                        // ParticleRng resource (particles.rs:128)
    std::array<ParticleRng, SlotRing::kMaxSlots> slot_rng{};  // its per-snapshot clones
    // content versions of the passive planes (BGR_CFG_SKIP_UNCHANGED_PLANES): equal ids <=> identical bytes
    uint64_t live_passive_ver = 1, ver_counter = 1;
    std::array<uint64_t, SlotRing::kMaxSlots> slot_passive_ver{};  // 0 = never written
};

struct Pending {
    uint32_t buf = 0;
    uint32_t chains = 1;            // result blocks to wait for
    unsigned long long seq = 0;
    unsigned long long gseq = 0;    // shard group sequence number (0: not in a group)
    bool finished = false;          // the GPU work is known to be complete (drain() synchronised the stream)
    uint32_t n_saves = 0;
    int32_t frames[kMaxSaves];
    uint32_t totals[kMaxSaves];
};

float duration_as_secs_f32(uint64_t ns) {  // core::time::Duration::as_secs_f32
    uint64_t secs = ns / 1000000000ULL;
    uint32_t nanos = uint32_t(ns % 1000000000ULL);
    return float(secs) + float(nanos) / 1000000000.0f;
}
uint32_t f32_bits(float f) { uint32_t b; std::memcpy(&b, &f, 4); return b; }

uint64_t host_ns() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return uint64_t(ts.tv_sec) * 1000000000ULL + uint64_t(ts.tv_nsec);
}

// The reference's tracing spans as NVTX ranges (no-ops unless a profiler is attached): `HandleRequests` around the
// whole call (schedule_systems.rs:171) and `SaveWorld` / `LoadWorld` / `AdvanceWorld` per request (:224-253) — around
// the host half of each request (ring push / rollback, frame resources, GgrsTime) while the vector is compiled, and
// around each request's kernel launches on the stepwise path.  On the fused paths the device half of all requests is
// ONE launch, which sits inside the HandleRequests range.
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};
inline const char* span_name(uint32_t request_kind) {
    return request_kind == BGR_REQ_SAVE ? "SaveWorld" : request_kind == BGR_REQ_LOAD ? "LoadWorld" : "AdvanceWorld";
}

int env_int(const char* name, int dflt) {
    const char* v = std::getenv(name);
    return v && *v ? std::atoi(v) : dflt;
}

}  // namespace

struct bgr_engine {
    bgr_config cfg{};
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int num_sms = 0;

    std::vector<Column> cols;
    std::vector<SystemReg> systems;
    uint32_t n_ck = 0;
    bool built = false;

    uint32_t epad = 0, words = 0, tile_bytes = 0, n_tiles_cap = 0;
    size_t image_bytes = 0;
    uint8_t* arena = nullptr;  // image 0 = live, image s+1 = slot s (tile-planar, kernels.cuh)
    uint8_t* d_kill = nullptr;
    uint8_t* d_stage = nullptr;  // device staging for ECS column <-> image transposition
    size_t stage_cap = 0;
    // asynchronous mirror downloads: packed on the main stream, copied D2H on copy_stream
    struct Download { uint8_t* d_buf = nullptr; size_t cap = 0; cudaEvent_t packed = nullptr, done = nullptr; bool busy = false; };
    Download dl[BGR_MAX_DOWNLOADS];
    cudaStream_t copy_stream = nullptr;
    uint32_t next_dl = 0;

    HostState st;

    static constexpr int kBufs = 8;  // result / spawn buffers = max un-collected submits (== PendingRing capacity)
    static constexpr int kMaxChains = 8;
    // Chains: the entity range is cut into n_chains contiguous tile ranges, each with its own stream, accumulators
    // and result block.  Entities are independent, so chain A's kernel of tick i+1 only depends on chain A's kernel
    // of tick i: with back-to-back submits the ramp / tail of one chain's kernel overlaps the other chain's kernel
    // (the same entity-range sharding as across GPUs, inside one GPU; partials are XOR-folded on the host).
    int n_chains = 1;
    cudaStream_t chain_stream[kMaxChains] = {};
    cudaEvent_t chain_ev[kMaxChains] = {};
    cudaEvent_t main_ev = nullptr;
    bool main_dirty = false;        // the main stream has un-synchronised work the chains must wait for
    uint32_t last_total_tiles = 0, last_chains = 0;  // tile partition of the previous chained launch
    unsigned long long* d_accum_c[kMaxChains] = {};
    unsigned int* d_ticket_c[kMaxChains] = {};
    unsigned long long* d_accum = nullptr;
    unsigned int* d_ticket = nullptr;
    float2* h_spawn[kBufs] = {};  // host-mapped (vx, vy) of spawned particles
    float2* d_spawn[kBufs] = {};
    int spawn_sys = -1;             // index of BGR_SYS_PARTICLES_SPAWN in `systems`, or -1
    unsigned long long* h_out[kBufs] = {};
    unsigned long long* d_out[kBufs] = {};
    cudaEvent_t ev[kBufs] = {};
    // un-collected request vectors, oldest first: a fixed ring (a std::deque allocated a chunk per push — the hot path
    // allocates nothing)
    struct PendingRing {
        Pending slot[8];
        uint32_t head = 0, count = 0;
        bool empty() const { return count == 0; }
        size_t size() const { return count; }
        void push_back(const Pending& p) { slot[(head + count) % 8u] = p; ++count; }
        Pending& front() { return slot[head]; }
        void pop_front() { head = (head + 1u) % 8u; --count; }
        template <class F> void for_each(F f) { for (uint32_t i = 0; i < count; ++i) f(slot[(head + i) % 8u]); }
    } pending;
    uint32_t next_buf = 0;
    std::vector<bgr_partial> last_partials;

    // shard group (multi-GPU): result blocks live in a shared host segment every rank's GPU and CPU map
    ShardGroup* group = nullptr;
    unsigned long long gseq = 0;
    unsigned long long* own_h_out[kBufs] = {};  // the engine's private result blocks while it is in a group
    unsigned long long* own_d_out[kBufs] = {};
    bool ticked = false;            // a request vector has been executed (the initial population is over)
    // device-side launch trace (bgr_trace_enable): per launch [first block start, last block end] in globaltimer ns
    unsigned long long* d_trace = nullptr;
    uint32_t trace_cap = 0;
    unsigned long long trace_first_seq = 0;

    uint64_t launches = 0;
    uint64_t prof[8] = {};          // host-side time of the hot loop: [0] calls, [1] compile ns, [2] launch ns, [3] wait ns, [4] fold ns
    bool last_fused = false;
    unsigned long long seq = 0;   // sequence number of the last submit (completion flag value)
    int tune_poll = 1;            // collect() spins on the host-mapped flag before falling back to the event
    int tune_tiledep = 1;         // consecutive fused launches overlap: per-tile dependencies instead of grid-level (PF_TILE_WAIT)
    unsigned int* d_tile_done = nullptr;  // [tiles] see ProgramParams::tile_done
    unsigned int* d_tile_cnt = nullptr;
    bool tiledep_chain = false;   // the last operation enqueued on the main stream was a PF_TILE_SIGNAL launch
    uint32_t tiledep_seq = 0, tiledep_tiles = 0;
    int tune_grid = 0;            // experiment / tests: cap the one-launch kernels' grid (0 = SMs x resident blocks)
    int tune_prefetch = 1;        // L2 prefetch of the next tile's active planes
    int tune_pdl = 0;             // programmatic dependent launch between consecutive fused kernels (measured: +0.8 % at 1M, -14 % at 100k -> off)
    int tune_dynamic = 1;         // dynamic tile scheduling in the fused kernel (measured +5% over a static stride)

    // compiled bundle: particles (update_particles + despawn_particles)
    bool bundle_particles = false;
    uint32_t bt = 0, bv = 0, bl = 0;
    std::vector<uint16_t> passive;
    std::vector<PassiveRun> runs;
    uint32_t passive_bytes = 0;
    bool bundle_static_ck = false;  // both columns checksummed with the finite assertion: fully specialised kernel
    // generic one-launch program (generic_program.cuh): any schema whose tile fits shared memory + the compiled systems
    bool generic_ok = false;
    int generic_bps[4] = {0, 0, 0, 0};  // resident blocks per SM of k_generic_program<64 | 128 | 256 | 512> (occupancy query, cached)
    int tune_jit = 1;               // 0 never, 1 worlds of >= 16k entities, 2 always: NVRTC-specialised generic program (jit.hpp)
    int tune_jit_rows = 4;          // rows of a tile per thread in the specialised kernel (1, 2, 4; measured: scripts/gpu_jit.sh)
    JitKernel jit;                  // fn == nullptr: the interpreter kernel runs.  Work item = a whole tile
    JitKernel jit_small;            // the same kernel with quarter-tile work items: worlds of few tiles per SM (optional)
    int tune_jit_tiledep = 0;       // 1: consecutive launches of the generated kernel overlap through per-item dependencies (queued submits)
    unsigned int* d_item_done = nullptr;   // [4 * tiles] GenericParams::item_done (quarter-tile work items at most)
    const void* jit_chain_kernel = nullptr;  // the signalling launch `tiledep_chain` refers to (its work-item partition must match)
    int tune_jit_item = 0;          // 0 auto (quarter tiles below 3 tiles per SM), 512 / 256 / 128 force the rows per work item
    int tune_generic_block = 0;     // 0 = 128; 64 / 256 / 512 force
    int tune_passive_early = -1;    // -1: early passive stores for single-wave grids (auto); 0 never; 1 always
    int tune_sub = 0;               // 128: the 128-row work-item variant of the fused kernel (experiment; default: whole tiles)
    int tune_stagger_ns = 800;      // start-of-grid phase stagger between the resident blocks of an SM (synchronous launches; measured -1.3 %)
    int tune_generic = 1;
    int tune_bundle = 1;            // 0: never use the specialised particles kernel (A/B tests of the generic program)
    bool bundle_opt = false;        // a registered column is BGR_STRATEGY_OPTIONAL: the presence-aware kernel variant (MODE 2)
    int tune_vec = 2, tune_minb = 2, tune_bps = 0, tune_passive_tma = 1;
    int tune_tma = 1;          // stepwise Save/Load through the TMA-staged bulk-copy kernel
    uint32_t tma_stage_tiles = 0;  // one-tile stages of the TMA copy kernel (0: schema too wide for two stages of shared memory)
    unsigned int* d_tma_ticket = nullptr;
    int occ_cache[2][3][3][3] = {};

    uint8_t* image(uint32_t idx) const { return arena + size_t(idx) * image_bytes; }
    uint32_t image_off256(uint32_t idx) const { return uint32_t((size_t(idx) * image_bytes) >> 8); }
    uint32_t tiles_for(uint32_t rows) const { return (rows + kTileRows - 1) / kTileRows; }
    uint32_t grid_for(uint32_t n, uint32_t per_block) const {
        uint32_t need = (n + per_block - 1) / per_block;
        uint32_t cap = uint32_t(num_sms) * 8u;
        return std::max(1u, std::min(need, cap));
    }
};

namespace {

// ---------------------------------------------------------------------------------------------
// compile: requests -> ops, mutating `s` exactly like handle_requests mutates the World
// ---------------------------------------------------------------------------------------------
struct Program {
    Op ops[kMaxOps];
    int32_t adv_frame[kMaxOps] = {};  // ADVANCE: RollbackFrameCount inside AdvanceWorld
    uint32_t n_ops = 0, n_saves = 0;
    int32_t save_frames[kMaxSaves];
    uint32_t save_totals[kMaxSaves];
    uint32_t max_rows = 0, live_rows = 0;
    bool has_load = false, has_advance = false, first_is_load = false, has_spawn = false;
    bool passive_to_slots = false;   // at least one SAVE must (re)write the passive planes
    bool passive_to_live = false;    // a LOAD changed the content of the live passive planes
    std::vector<float2> spawn_vals;
};

int compile_requests(bgr_engine* e, HostState& s, const bgr_session_info* sess, const bgr_request* reqs, uint32_t n,
                     Program& pg) {
    if (n > kMaxOps) return fail(BGR_ERR_CAPACITY, "too many requests in one handle_requests call");
    pg.live_rows = s.n_rows;
    pg.max_rows = s.n_rows;
    uint32_t n_counter_systems = 0;
    for (auto& sy : e->systems) n_counter_systems += (sy.id == BGR_SYS_U32_STORE_CALL_COUNT);
    for (uint32_t i = 0; i < n; ++i) {
        const bgr_request& rq = reqs[i];
        NvtxRange span(span_name(rq.kind));
        // schedule_systems.rs:190-220 — resources recomputed from the session before every request
        const int32_t current_frame = s.frame_count;
        if (sess) {
            switch (sess->kind) {
            case BGR_SESSION_P2P:
                s.has_maxpred = true; s.maxpred = sess->max_prediction;
                s.confirmed = sess->confirmed_frame;
                break;
            case BGR_SESSION_SYNCTEST: {
                s.has_maxpred = true; s.maxpred = sess->max_prediction;
                int32_t cf = current_frame - int32_t(sess->check_distance);
                if (cf >= 0) s.confirmed = cf;
                break;
            }
            case BGR_SESSION_SPECTATOR:
                s.has_maxpred = true; s.maxpred = 0;
                s.confirmed = current_frame;
                break;
            default: break;
            }
        }
        Op& op = pg.ops[pg.n_ops];
        std::memset(&op, 0, sizeof op);
        switch (rq.kind) {
        case BGR_REQ_SAVE: {  // :223-237 -> SaveWorld: sync_depth, discard_old_snapshots, save (component_snapshot.rs:135-144)
            if (pg.n_saves >= kMaxSaves) return fail(BGR_ERR_CAPACITY, "too many SaveGameState requests in one call");
            if (s.has_maxpred) s.ring.set_depth(s.maxpred);
            s.ring.confirm(s.confirmed);
            uint32_t slot = s.ring.push(s.frame_count);
            if (slot == SlotRing::kNoSlot)
                return fail(BGR_ERR_CAPACITY, "snapshot ring needs more frame slots than bgr_config.max_depth");
            op.kind = OP_SAVE;
            if (slot == SlotRing::kNoSlot - 1) { op.flags |= OPF_NO_STORE; op.image_off256 = 0; }
            else {
                op.image_off256 = e->image_off256(slot + 1);
                s.slot_rows[slot] = s.n_rows;
                s.slot_elapsed_ns[slot] = s.elapsed_ns;
                s.slot_rng[slot] = s.rng;
                if ((e->cfg.flags & BGR_CFG_SKIP_UNCHANGED_PLANES) && s.slot_passive_ver[slot] == s.live_passive_ver)
                    op.flags |= OPF_SKIP_PASSIVE;
                else
                    pg.passive_to_slots = true;
                s.slot_passive_ver[slot] = s.live_passive_ver;
            }
            op.n_rows = s.n_rows;
            op.save_index = pg.n_saves;
            pg.save_frames[pg.n_saves] = rq.frame;
            pg.save_totals[pg.n_saves] = s.n_rows;
            ++pg.n_saves;
            break;
        }
        case BGR_REQ_LOAD: {  // :238-250 -> LoadWorld
            s.frame_count = rq.frame;
            std::string err;
            if (!s.ring.rollback(rq.frame, &err)) return fail(BGR_ERR_NO_SNAPSHOT, err);
            uint32_t slot = 0;
            if (!s.ring.get(&slot, &err)) return fail(BGR_ERR_NO_SNAPSHOT, err);
            s.n_rows = s.slot_rows[slot];
            s.elapsed_ns = s.slot_elapsed_ns[slot];
            s.rng = s.slot_rng[slot];
            if (!(e->cfg.flags & BGR_CFG_SKIP_UNCHANGED_PLANES) || s.slot_passive_ver[slot] != s.live_passive_ver)
                pg.passive_to_live = true;
            s.live_passive_ver = s.slot_passive_ver[slot];
            op.kind = OP_LOAD;
            op.image_off256 = e->image_off256(slot + 1);
            op.n_rows = s.n_rows;
            if (pg.n_ops == 0) pg.first_is_load = true;
            pg.has_load = true;
            break;
        }
        case BGR_REQ_ADVANCE:
        case kReqAdvanceNoBump: {  // :251-269 -> AdvanceWorld
            if (rq.kind == BGR_REQ_ADVANCE) s.frame_count += 1;
            if (rq.n_players > BGR_MAX_PLAYERS) return fail(BGR_ERR_INVALID_ARGUMENT, "n_players > BGR_MAX_PLAYERS");
            // GgrsTimePlugin::update (time.rs:63-76): advance_to(frame * 1e9 / fps)
            uint64_t runtime = uint64_t(int64_t(s.frame_count)) * 1000000000ULL / uint64_t(e->cfg.fps);
            if (runtime < s.elapsed_ns)
                return fail(BGR_ERR_STATE, "tried to move Time<GgrsTime> backwards (RollbackFrameCount went back without LoadWorld)");
            uint64_t delta = runtime - s.elapsed_ns;
            s.elapsed_ns = runtime;
            op.kind = OP_ADVANCE;
            pg.adv_frame[pg.n_ops] = s.frame_count;
            op.dt_bits = f32_bits(duration_as_secs_f32(delta));
            op.n_rows = s.n_rows;
            op.call_count = s.call_count;
            s.call_count += n_counter_systems;
            for (uint32_t k = 0; k < BGR_MAX_PLAYERS && k < rq.n_players; ++k) op.inputs[k] = rq.inputs[k];
            op.flags |= (rq.n_players & 0xFu) << 8;  // PlayerInputs<T>.len() for systems that index it (box_game.rs:171)
            pg.has_advance = true;
            if (e->spawn_sys >= 0) {  // spawn_particles.run_if(spawn_pressed) (particles.rs:236, 254-256)
                bool pressed = false;
                for (uint32_t k = 0; k < rq.n_players; ++k) pressed = pressed || (rq.inputs[k] & BGR_INPUT_SPAWN);
                if (pressed) {
                    const SystemReg& sy = e->systems[size_t(e->spawn_sys)];
                    const uint32_t rate = sy.params[0];
                    if (uint64_t(s.n_rows) + rate > e->cfg.max_entities)
                        return fail(BGR_ERR_CAPACITY, "spawn_particles exceeds max_entities");
                    if (pg.spawn_vals.size() + rate > kMaxSpawnVals)
                        return fail(BGR_ERR_CAPACITY, "too many particles spawned by one request vector");
                    op.flags |= OPF_SPAWN;
                    op.image_off256 = s.n_rows;                      // first spawned row
                    op.save_index = rate;                            // count
                    op.call_count = uint32_t(pg.spawn_vals.size());  // offset into spawn_vals
                    for (uint32_t k = 0; k < rate; ++k) {            // particles.rs:262-268
                        float2 v;
                        v.x = s.rng.random_range(-200.0f, 200.0f);
                        v.y = s.rng.random_range(-200.0f, 200.0f);
                        pg.spawn_vals.push_back(v);
                    }
                    s.n_rows += rate;  // Rollback on_add -> RollbackOrdered.push, applied at the end of the frame
                    s.live_passive_ver = ++s.ver_counter;  // newborn rows carry Transform::default() rotation / scale
                    pg.has_spawn = true;
                    pg.max_rows = std::max(pg.max_rows, s.n_rows);
                }
            }
            break;
        }
        default: return fail(BGR_ERR_INVALID_ARGUMENT, "unknown request kind");
        }
        pg.max_rows = std::max(pg.max_rows, op.n_rows);
        ++pg.n_ops;
    }
    return BGR_OK;
}

// ---------------------------------------------------------------------------------------------
// launch: fused bundle kernel
// ---------------------------------------------------------------------------------------------
template <int VEC, int MODE, int MINB, int SUB = int(kTileRows)>
int launch_particles(bgr_engine* e, const ProgramParams& pp, int vi, int si, int mi, cudaStream_t stream) {
    auto kern = k_particles_program<VEC, MODE, MINB, SUB>;
    constexpr int BLOCK = SUB / VEC;
    constexpr uint32_t kSubs = kTileRows / SUB;
    constexpr int ui = kSubs > 1 ? 1 : 0;
    const size_t smem = (pp.flags & PF_PASSIVE_TMA) ? size_t(2) * pp.passive_bytes : 0;
    if (e->occ_cache[ui][vi][si][mi] == 0) {
        if (smem > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
        int nb = 0;
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, BLOCK, smem));
        e->occ_cache[ui][vi][si][mi] = std::max(1, nb);
    }
    int bps = e->occ_cache[ui][vi][si][mi];
    if (e->tune_bps > 0) bps = std::min(e->tune_bps, bps);
    uint32_t grid = std::max(1u, std::min((pp.n_tiles - pp.tile_begin) * kSubs, uint32_t(e->num_sms * bps)));
    if (e->tune_grid > 0) grid = std::min(grid, uint32_t(e->tune_grid));
    if (kSubs > 1) grid = std::max(kSubs, grid / kSubs * kSubs);  // the first wave covers whole tiles (per-tile completion counts)
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(grid); lc.blockDim = dim3(BLOCK); lc.dynamicSmemBytes = smem; lc.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    const bool pdl = e->tune_pdl || (pp.flags & PF_TILE_WAIT);
    lc.attrs = attr; lc.numAttrs = pdl ? 1 : 0;
    CUDA_TRY(cudaLaunchKernelEx(&lc, kern, pp));
    CUDA_TRY(cudaGetLastError());
    e->launches += 1;
    return BGR_OK;
}

int launch_fused_variant(bgr_engine* e, const ProgramParams& pp, cudaStream_t stream);

int run_fused(bgr_engine* e, const Program& pg, uint32_t buf, uint32_t* chains_out) {
    ProgramParams pp;
    std::memset(&pp, 0, sizeof pp);
    pp.seq = e->seq;
    pp.arena = e->arena;
    pp.order_base = e->cfg.order_base;
    pp.words = e->words; pp.tile_bytes = e->tile_bytes;
    const uint32_t total_tiles = std::max(1u, e->tiles_for(pg.max_rows));  // at least one tile so a result block is published
    pp.n_ops = pg.n_ops; pp.n_saves = pg.n_saves;
    pp.live_rows = pg.live_rows;
    pp.flags = 0;
    if (!pg.first_is_load) pp.flags |= PF_READ_LIVE;
    if (pg.has_load || pg.has_advance) pp.flags |= PF_WRITE_LIVE_ACTIVE;
    if ((pg.has_load && pg.passive_to_live) || pg.has_spawn) pp.flags |= PF_WRITE_LIVE_PASSIVE;
    const bool passive_needed = pg.passive_to_slots || (pp.flags & PF_WRITE_LIVE_PASSIVE) || pg.has_spawn;
    uint32_t n_loads = 0;
    for (uint32_t i = 0; i < pg.n_ops; ++i) n_loads += (pg.ops[i].kind == OP_LOAD);
    const bool simple = n_loads == 0 || (n_loads == 1 && pg.first_is_load);
    if (e->tune_dynamic) pp.flags |= PF_DYNAMIC_TILES;
    if (e->tune_prefetch) pp.flags |= PF_PREFETCH_NEXT;
    pp.spawn_vals = e->d_spawn[buf];
    if (e->spawn_sys >= 0) {
        const uint64_t ttl = e->systems[size_t(e->spawn_sys)].params[1];
        pp.spawn_ttl_lo = uint32_t(ttl); pp.spawn_ttl_hi = uint32_t(ttl >> 32);
    }
    if (!pg.has_spawn && simple && e->tune_passive_tma && !e->runs.empty() && 2u * e->passive_bytes <= 96u * 1024u) pp.flags |= PF_PASSIVE_TMA;
    // Opt-in experiment (BGR_TUNE_SUB=128): cut every tile into 128-row work items handled by 64-thread blocks
    // (kernels.cuh `SUB`).  Meant to balance small worlds (100k entities = 196 tiles on 148 SMs); measured SLOWER there
    // (21.2 vs 17.2 us per tick): the better balance is paid for with fewer warps per scheduler on the busy SMs and
    // per-plane bulk copies, and the tick is issue-latency-bound on the hash, not imbalance-bound.  Kept for A/B runs.
    const bool sub_items = e->tune_sub == 128;
    if (sub_items && e->tune_vec == 2 && e->n_chains == 1) pp.flags |= PF_SUB_ITEMS;
    // one wave of blocks (every block runs one or two tiles): the tile's tail is the grid's tail
    if (e->tune_passive_early == 1 || (e->tune_passive_early < 0 && total_tiles <= 3u * uint32_t(e->num_sms))) pp.flags |= PF_PASSIVE_EARLY;
    const Column& ct = e->cols[e->bt]; const Column& cv = e->cols[e->bv];
    if (ct.hash_kind != BGR_HASH_NONE) { pp.flags |= PF_CK_T; if (ct.hash_flags & BGR_HASH_FLAG_ASSERT_FINITE_F32) pp.flags |= PF_FIN_T; pp.ck_t_slot = uint32_t(ct.ck_slot); }
    if (cv.hash_kind != BGR_HASH_NONE) { pp.flags |= PF_CK_V; if (cv.hash_flags & BGR_HASH_FLAG_ASSERT_FINITE_F32) pp.flags |= PF_FIN_V; pp.ck_v_slot = uint32_t(cv.ck_slot); }
    pp.t_off = ct.first_plane * kPlaneBytes; pp.v_off = cv.first_plane * kPlaneBytes;
    pp.l_off = e->cols[e->bl].first_plane * kPlaneBytes; pp.alive_off = e->words * kPlaneBytes;
    pp.need_t = ct.absent; pp.need_v = cv.absent; pp.need_tv = ct.absent | cv.absent; pp.need_l = e->cols[e->bl].absent;
    pp.n_runs = passive_needed ? uint32_t(e->runs.size()) : 0u;
    pp.passive_bytes = (pp.flags & PF_SUB_ITEMS) ? uint32_t(e->passive.size()) * 128u * 4u : e->passive_bytes;
    for (size_t i = 0; i < e->runs.size(); ++i) pp.runs[i] = e->runs[i];
    pp.n_passive = passive_needed ? uint32_t(e->passive.size()) : 0u;
    for (size_t i = 0; i < e->passive.size(); ++i) {
        pp.passive[i] = e->passive[i];
        // Transform::default(): rotation = (0,0,0,1), scale = (1,1,1); every other passive word of a newborn row is 0
        const uint32_t tw = uint32_t(e->passive[i]) - ct.first_plane;
        pp.passive_template[i] = (uint32_t(e->passive[i]) >= ct.first_plane && tw >= 6 && tw <= 9) ? 0x3f800000u : 0u;
    }
    std::memcpy(pp.ops, pg.ops, sizeof(Op) * pg.n_ops);

    // one launch per chain: contiguous tile ranges, own stream / accumulators / result block
    const uint32_t chains = std::max(1u, std::min(uint32_t(e->n_chains), total_tiles));
    *chains_out = chains;
    // Chain c of this launch follows chain c of the previous one in stream order, which is all the ordering the data
    // needs while both cover the same tiles.  A changed partition (rows spawned, first launch), stepwise work, or a
    // caller-owned stream (whose earlier work we cannot see) makes every chain wait for everything before it.
    if (chains != e->last_chains || total_tiles != e->last_total_tiles || !e->own_stream) e->main_dirty = true;
    e->last_chains = chains; e->last_total_tiles = total_tiles;
    if (chains > 1 && e->main_dirty) {
        CUDA_TRY(cudaEventRecord(e->main_ev, e->stream));
        for (uint32_t c = 0; c < chains; ++c) CUDA_TRY(cudaStreamWaitEvent(e->chain_stream[c], e->main_ev, 0));
        e->main_dirty = false;
    }
    // only worth it when request vectors are queued behind each other (bgr_submit_requests with others un-collected):
    // a synchronous caller collects before the next submit, so there is nothing to overlap with
    // ... and only on a stream the engine owns: on a caller's stream foreign work may sit between two submits and
    // become the programmatic-launch primary, which the per-tile flags know nothing about
    const bool tiledep = e->tune_tiledep && chains == 1 && e->d_tile_done && e->own_stream && (e->tune_tiledep > 1 || !e->pending.empty());
    if (e->tiledep_chain && total_tiles != e->tiledep_tiles) {
        // The tile range changed (rows crossed a tile boundary): a tile outside the previous launch's range may still be
        // in use by an OLDER overlapping launch that nothing would make this one wait for.  Rare: drain the stream.
        CUDA_TRY(cudaStreamSynchronize(e->stream));
        e->tiledep_chain = false;
    }
    if (tiledep) {
        pp.flags |= PF_TILE_SIGNAL;
        pp.grid_done = e->d_tile_done + e->tiles_for(e->cfg.max_entities);  // the extra word behind the per-tile flags
        pp.tile_done = e->d_tile_done; pp.tile_cnt = e->d_tile_cnt;
        pp.done_seq = uint32_t(e->seq);
        if (e->tiledep_chain) { pp.flags |= PF_TILE_WAIT; pp.wait_seq = e->tiledep_seq; pp.wait_tiles = e->tiledep_tiles; }
    }
    // start stagger: only launches that start on an idle GPU with at least two resident blocks per SM (overlapping
    // launches arrive dephased already)
    if (e->tune_stagger_ns > 0 && !(pp.flags & PF_TILE_WAIT) && total_tiles / chains >= 2u * uint32_t(e->num_sms)) {
        pp.stagger_ns = uint32_t(e->tune_stagger_ns); pp.stagger_div = uint32_t(e->num_sms);
    }
    for (uint32_t c = 0; c < chains; ++c) {
        pp.tile_begin = uint32_t(uint64_t(total_tiles) * c / chains);
        pp.n_tiles = uint32_t(uint64_t(total_tiles) * (c + 1) / chains);
        // overlapping launches (tile dependencies) must not share accumulators / tickets: rotate over kBufs sets — at
        // most kBufs request vectors are un-collected, so a set is re-armed (before its launch's completion word is
        // written) long before the launch kBufs later touches it
        static_assert(bgr_engine::kMaxChains >= bgr_engine::kBufs, "one accumulator set per in-flight request vector");
        const uint32_t set = tiledep ? uint32_t(e->seq % bgr_engine::kBufs) : c;
        pp.accum = e->d_accum_c[set];
        pp.ticket = e->d_ticket_c[set];
        pp.out = e->d_out[buf] + size_t(c) * kResultStride;
        pp.trace = nullptr;
        if (e->d_trace && c == 0 && e->seq - e->trace_first_seq < e->trace_cap) pp.trace = e->d_trace + (e->seq - e->trace_first_seq) * 4;
        cudaStream_t stream = chains > 1 ? e->chain_stream[c] : e->stream;
        int rc = launch_fused_variant(e, pp, stream);
        if (rc != BGR_OK) return rc;
        if (chains > 1) {  // everything later on the main stream (and external timing events) is ordered after the chains
            CUDA_TRY(cudaEventRecord(e->chain_ev[c], stream));
            CUDA_TRY(cudaStreamWaitEvent(e->stream, e->chain_ev[c], 0));
        }
    }
    e->tiledep_chain = tiledep;
    e->tiledep_seq = uint32_t(e->seq); e->tiledep_tiles = total_tiles;
    return BGR_OK;
}

int launch_fused_variant(bgr_engine* e, const ProgramParams& pp, cudaStream_t stream) {
    const int v = e->bundle_opt ? 2 : e->tune_vec;
    const bool st = e->bundle_static_ck && !e->bundle_opt;
    if (pp.flags & PF_SUB_ITEMS) {  // small worlds: 128-row work items, 64-thread blocks, 768 threads per SM
        constexpr int kSub = 128, kMinbSub = 768 / (kSub / 2);
        if (e->bundle_opt) return launch_particles<2, 2, kMinbSub, kSub>(e, pp, 1, 2, 1, stream);
        if (st) return launch_particles<2, 1, kMinbSub, kSub>(e, pp, 1, 1, 1, stream);
        return launch_particles<2, 0, kMinbSub, kSub>(e, pp, 1, 0, 1, stream);
    }
    const int mb = e->tune_minb >= 8 ? 2 : (e->tune_minb >= 2 ? 1 : 0);  // launch-bounds tier: 1024 / 768 / unconstrained threads per SM
    if (e->bundle_opt) {  // per-entity presence: one variant (2 rows per thread, 768 threads per SM)
        constexpr int kMidOpt = 768 / int(kTileRows / 2);
        return launch_particles<2, 2, kMidOpt>(e, pp, 1, 2, 1, stream);
    }
#define BGR_LAUNCH(VEC, VI)                                                                                \
    if (v == VEC) {                                                                                        \
        constexpr int kHi = (1024 / int(kTileRows / VEC)) > 32 ? 32 : (1024 / int(kTileRows / VEC));        \
        constexpr int kMid = (768 / int(kTileRows / VEC)) < 1 ? 1 : (768 / int(kTileRows / VEC));           \
        if (st && mb == 2) return launch_particles<VEC, 1, kHi>(e, pp, VI, 1, 2, stream);                          \
        if (st && mb == 1) return launch_particles<VEC, 1, kMid>(e, pp, VI, 1, 1, stream);                         \
        if (st) return launch_particles<VEC, 1, 1>(e, pp, VI, 1, 0, stream);                                       \
        if (mb == 2) return launch_particles<VEC, 0, kHi>(e, pp, VI, 0, 2, stream);                                \
        if (mb == 1) return launch_particles<VEC, 0, kMid>(e, pp, VI, 0, 1, stream);                               \
        return launch_particles<VEC, 0, 1>(e, pp, VI, 0, 0, stream);                                               \
    }
    BGR_LAUNCH(1, 0)
    BGR_LAUNCH(4, 2)
    BGR_LAUNCH(2, 1)
#undef BGR_LAUNCH
    return fail(BGR_ERR_STATE, "bad BGR_TUNE_VEC");
}

// ---------------------------------------------------------------------------------------------
// launch: TMA-staged image copy (+ fused checksum for a Save)
// ---------------------------------------------------------------------------------------------
int launch_tma(bgr_engine* e, const uint8_t* src, uint8_t* dst, uint32_t n_rows_src, uint32_t n_rows_copy, bool save,
               unsigned long long* acc, bool store) {
    TmaCopyParams tp;
    std::memset(&tp, 0, sizeof tp);
    tp.src = src; tp.dst = dst;
    tp.order_base = e->cfg.order_base;
    tp.accum = save ? acc : nullptr;
    tp.words = e->words; tp.tile_bytes = e->tile_bytes; tp.stages = e->tma_stage_tiles;
    tp.ticket = e->d_tma_ticket;
    tp.n_tiles = e->tiles_for(n_rows_copy);
    tp.n_rows_src = n_rows_src;
    tp.count_alive = save ? 1u : 0u;
    tp.store = store ? 1u : 0u;
    if (save)
        for (const Column& c : e->cols)
            if (c.hash_kind != BGR_HASH_NONE) {
                HashSpec& h = tp.hash[tp.n_hash++];
                h.first_plane = c.first_plane; h.off = c.hash_off; h.len = c.hash_len;
                h.finite = c.hash_flags & BGR_HASH_FLAG_ASSERT_FINITE_F32; h.slot = uint32_t(c.ck_slot);
                h.absent = c.absent;
            }
    uint32_t grid = std::max(1u, std::min(tp.n_tiles, uint32_t(e->num_sms)));
    size_t smem = size_t(tp.stages) * e->tile_bytes;
    k_image_tma<<<grid, kTmaBlock, smem, e->stream>>>(tp);
    CUDA_TRY(cudaGetLastError());
    e->launches += 1;
    return BGR_OK;
}

// ---------------------------------------------------------------------------------------------
// launch: stepwise path (generic schemas / systems)
// ---------------------------------------------------------------------------------------------
int run_stepwise(bgr_engine* e, const Program& pg, uint32_t buf) {
    e->main_dirty = true;
    e->tiledep_chain = false;
    uint32_t live_rows = pg.live_rows;
    uint8_t* live = e->image(0);
    for (uint32_t i = 0; i < pg.n_ops; ++i) {
        const Op& op = pg.ops[i];
        NvtxRange span(span_name(op.kind == OP_SAVE ? uint32_t(BGR_REQ_SAVE) : op.kind == OP_LOAD ? uint32_t(BGR_REQ_LOAD) : uint32_t(BGR_REQ_ADVANCE)));
        switch (op.kind) {
        case OP_SAVE: {
            unsigned long long* acc = e->d_accum + size_t(op.save_index) * kAccStride;
            if (e->tune_tma && e->tma_stage_tiles) {
                int rc = launch_tma(e, live, e->arena + (size_t(op.image_off256) << 8), op.n_rows, op.n_rows, true, acc, !(op.flags & OPF_NO_STORE));
                if (rc != BGR_OK) return rc;
                break;
            }
            bool counted = false;
            for (const Column& c : e->cols) {
                if (c.hash_kind == BGR_HASH_NONE) continue;
                k_checksum_column<<<e->grid_for(std::max(1u, op.n_rows), 256), 256, 0, e->stream>>>(
                    live, e->words, c.first_plane, c.hash_off, c.hash_len,
                    c.hash_flags & BGR_HASH_FLAG_ASSERT_FINITE_F32, op.n_rows, e->cfg.order_base, acc,
                    uint32_t(c.ck_slot), counted ? 0u : 1u, 1u, c.absent);
                counted = true;
                e->launches += 1;
            }
            if (!counted) {
                k_checksum_column<<<e->grid_for(std::max(1u, op.n_rows), 256), 256, 0, e->stream>>>(
                    live, e->words, 0, 0, 0, 0, op.n_rows, e->cfg.order_base, acc, 0, 1u, 0u, 0u);
                e->launches += 1;
            }
            if (!(op.flags & OPF_NO_STORE) && op.n_rows > 0) {
                uint32_t nt = e->tiles_for(op.n_rows);
                k_copy_image<<<e->grid_for(uint32_t(size_t(nt) * e->tile_bytes / 16u), 256), 256, 0, e->stream>>>(
                    live, e->arena + (size_t(op.image_off256) << 8), e->words, nt, op.n_rows);
                e->launches += 1;
            }
            break;
        }
        case OP_LOAD: {
            uint32_t n_copy = std::max(op.n_rows, live_rows);
            if (n_copy > 0 && e->tune_tma && e->tma_stage_tiles) {
                int rc = launch_tma(e, e->arena + (size_t(op.image_off256) << 8), live, op.n_rows, n_copy, false, nullptr, true);
                if (rc != BGR_OK) return rc;
            } else if (n_copy > 0) {
                uint32_t nt = e->tiles_for(n_copy);
                k_copy_image<<<e->grid_for(uint32_t(size_t(nt) * e->tile_bytes / 16u), 256), 256, 0, e->stream>>>(
                    e->arena + (size_t(op.image_off256) << 8), live, e->words, nt, op.n_rows);
                e->launches += 1;
            }
            live_rows = op.n_rows;
            break;
        }
        case OP_ADVANCE: {
            bool any_despawn = false;
            uint32_t counter = op.call_count;
            uint32_t n = op.n_rows;
            uint32_t grid = e->grid_for(std::max(1u, n), 256);
            for (const SystemReg& sy : e->systems) {
                if (n == 0) break;
                uint32_t need = 0;  // the query matches entities that have every bound column
                for (uint32_t c : sy.cols) need |= e->cols[c].absent;
                switch (sy.id) {
                case BGR_SYS_PARTICLES_UPDATE:
                    k_sys_particles_update<<<grid, 256, 0, e->stream>>>(live, e->words, e->cols[sy.cols[0]].first_plane,
                                                                          e->cols[sy.cols[1]].first_plane, n, op.dt_bits, need);
                    break;
                case BGR_SYS_PARTICLES_DESPAWN:
                    k_sys_particles_despawn<<<grid, 256, 0, e->stream>>>(live, e->words, e->cols[sy.cols[0]].first_plane, n, e->d_kill, need);
                    any_despawn = true;
                    break;
                case BGR_SYS_U32_ADD:
                    k_sys_u32_add<<<grid, 256, 0, e->stream>>>(live, e->words, e->cols[sy.cols[0]].first_plane + sy.params[0] / 4, n, sy.params[1], need);
                    break;
                case BGR_SYS_U32_SATSUB_DESPAWN:
                    k_sys_u32_satsub_despawn<<<grid, 256, 0, e->stream>>>(live, e->words, e->cols[sy.cols[0]].first_plane + sy.params[0] / 4, n, sy.params[1], e->d_kill, need);
                    any_despawn = true;
                    break;
                case BGR_SYS_U32_STORE_CALL_COUNT:
                    k_sys_u32_store<<<grid, 256, 0, e->stream>>>(live, e->words, e->cols[sy.cols[0]].first_plane + sy.params[0] / 4, n, counter++, need);
                    break;
                case BGR_SYS_PARTICLES_SPAWN:
                    continue;  // Commands: applied after the schedule (below)
                case BGR_SYS_DESPAWN_ON_INPUT: {
                    const uint32_t player = sy.params[0], n_players = (op.flags >> 8) & 0xFu;
                    const uint32_t input = player < n_players ? op.inputs[player] : 0u;
                    if (input != sy.params[1]) continue;  // the run condition is host-known: no launch on other frames
                    k_sys_despawn_having<<<grid, 256, 0, e->stream>>>(live, e->words, n, e->d_kill, need);
                    any_despawn = true;
                    break;
                }
                case BGR_SYS_BOX_MOVE: {
                    unsigned long long packed = 0;
                    for (int k = 0; k < 8; ++k) packed |= (unsigned long long)(op.inputs[k]) << (8 * k);
                    k_sys_box_move<<<grid, 256, 0, e->stream>>>(live, e->words, e->cols[sy.cols[0]].first_plane, e->cols[sy.cols[1]].first_plane,
                                                                 n, op.dt_bits, packed, (op.flags >> 8) & 0xFu, e->cfg.order_base, need);
                    break;
                }
                default: return fail(BGR_ERR_UNSUPPORTED, "system has no GPU implementation yet");
                }
                e->launches += 1;
            }
            if (any_despawn) {
                k_apply_despawns<<<grid, 256, 0, e->stream>>>(live, e->words, n, e->d_kill);
                e->launches += 1;
            }
            break;
        }
        default: break;
        }
        if (op.kind == OP_ADVANCE && (op.flags & OPF_SPAWN)) {
            const SystemReg& sy = e->systems[size_t(e->spawn_sys)];
            const uint64_t ttl = sy.params[1];
            k_sys_particles_spawn<<<e->grid_for(op.save_index, 256), 256, 0, e->stream>>>(
                live, e->words, e->cols[sy.cols[0]].first_plane, e->cols[sy.cols[1]].first_plane, e->cols[sy.cols[2]].first_plane,
                op.image_off256, op.save_index, e->d_spawn[buf] + op.call_count, uint32_t(ttl), uint32_t(ttl >> 32));
            e->launches += 1;
            live_rows = std::max(live_rows, op.image_off256 + op.save_index);
        }
    }
    k_publish<<<1, 128, 0, e->stream>>>(e->d_accum, e->d_out[buf], std::max(1u, pg.n_saves) * kAccStride, e->seq);
    e->launches += 1;
    CUDA_TRY(cudaGetLastError());
    return BGR_OK;
}


// the registration as the generic program's spec tables (parameter block of the interpreter, prelude of the JIT kernel)
void fill_generic_specs(const bgr_engine* e, GenericParams& gp) {
    gp.n_hash = 0;
    gp.n_sys = 0;
    for (const Column& c : e->cols)
        if (c.hash_kind != BGR_HASH_NONE) {
            HashSpec& h = gp.hash[gp.n_hash++];
            h.first_plane = c.first_plane; h.off = c.hash_off; h.len = c.hash_len;
            h.finite = c.hash_flags & BGR_HASH_FLAG_ASSERT_FINITE_F32; h.slot = uint32_t(c.ck_slot);
            h.absent = c.absent;
        }
    uint32_t counter_index = 0, user_index = 0;
    for (const SystemReg& sy : e->systems) {
        SysSpec& sp = gp.sys[gp.n_sys++];
        sp.id = sy.id;
        for (uint32_t c : sy.cols) sp.need |= e->cols[c].absent;
        sp.plane0 = e->cols[sy.cols[0]].first_plane;
        switch (sy.id) {
        case BGR_SYS_U32_ADD:
        case BGR_SYS_U32_SATSUB_DESPAWN: sp.plane0 += sy.params[0] / 4; sp.param = sy.params[1]; break;
        case BGR_SYS_U32_STORE_CALL_COUNT: sp.plane0 += sy.params[0] / 4; sp.param = counter_index++; break;
        case BGR_SYS_DESPAWN_ON_INPUT: sp.param = sy.params[0] | (sy.params[1] << 8); break;
        case BGR_SYS_PARTICLES_UPDATE:
        case BGR_SYS_BOX_MOVE: sp.plane1 = e->cols[sy.cols[1]].first_plane; break;
        case kSysUser: sp.param = user_index++; break;  // the planes are literals of its dispatcher (jit_specialise)
        default: break;
        }
    }
}

// A C string literal of `text` for a generated static_assert message.
std::string c_string_literal(const std::string& text) {
    std::string out = "\"";
    for (char ch : text) {
        if (ch == '"' || ch == '\\') out += '\\';
        out += (ch >= 0x20 && ch < 0x7f) ? ch : '?';
    }
    return out + "\"";
}

// The prelude's part for user systems: the device API, every source in its own namespace with its own line numbers, and
// one dispatcher per system that binds the function's parameters to the literal word planes of its columns.
std::string user_systems_prelude(const bgr_engine* e) {
    std::string pre = "#define BGR_SYS_USER " + std::to_string(kSysUser) + "\n#include \"user_system.cuh\"\n";
    uint32_t user_index = 0;
    for (const SystemReg& sy : e->systems) {
        if (sy.id != kSysUser) continue;
        const std::string idx = std::to_string(user_index++), ns = "bgr_user_" + idx, fn = ns + "::" + sy.name;
        pre += "namespace " + ns + " {\n#line 1 \"" + sy.name + "\"\n" + sy.source + "\n}\n";
        pre += "#line 1 \"bgr_user_dispatch_" + sy.name + "\"\n";
        pre += "template <> struct bgr_user_system<" + idx + "> {\n";
        pre += "    using F = bgr_fn_traits<decltype(&" + fn + ")>;\n";
        pre += "    static_assert(F::arity == " + std::to_string(sy.cols.size()) + ", " +
               c_string_literal(sy.name + ": takes one component parameter per bound column (" + std::to_string(sy.cols.size()) + ")") + ");\n";
        std::string planes;
        for (size_t i = 0; i < sy.cols.size(); ++i) {
            const Column& c = e->cols[sy.cols[i]];
            pre += "    static_assert(sizeof(F::elem<" + std::to_string(i) + ">) == " + std::to_string(c.elem_bytes) + ", " +
                   c_string_literal(sy.name + ": parameter " + std::to_string(i + 1) + " is bound to column '" + c.name + "' of " +
                                    std::to_string(c.elem_bytes) + " bytes; sizeof of the parameter type differs") + ");\n";
            planes += (i ? ", " : "") + std::to_string(c.first_plane);
        }
        pre += "    template <int N> static __device__ __forceinline__ void run(uint32_t (&w)[N], bool on, const bgr_sys_ctx& base, bool& kill) {\n";
        pre += "        bgr_sys_ctx ctx = base;\n";
        for (size_t j = 0; j < 8; ++j)
            pre += "        ctx.params[" + std::to_string(j) + "] = " + std::to_string(j < sy.params.size() ? sy.params[j] : 0u) + "u;\n";
        pre += "        bgr_invoke<&" + fn + ">::run<" + planes + ">(w, on, ctx, kill);\n    }\n};\n";
    }
    return pre;
}

// NVRTC specialisation of the generic program for this registration (jit.hpp, generic_program_jit.cuh); called by bgr_build.
// Registrations of compiled-in systems keep the interpreter when this fails (always BGR_OK).  A registration with user
// systems has no other kernel: every reason it cannot be compiled is an error of bgr_build.
int jit_specialise(bgr_engine* e) {
    e->jit = JitKernel{};
    e->jit_small = JitKernel{};
    const bool user = has_user_systems(e->systems);  // bgr_build has refused what user systems cannot run with
    if (!e->generic_ok || !e->tune_generic || e->tune_jit == 0 || (e->cfg.flags & BGR_CFG_FORCE_STEPWISE)) return BGR_OK;
    if (e->bundle_particles && e->tune_bundle) return BGR_OK;  // the bundle has its own kernel
    // small worlds: a tick is launch latency, not worth a compile (user systems run on nothing else)
    if (!user && e->tune_jit == 1 && e->cfg.max_entities < 16384) return BGR_OK;
    GenericParams gp;
    std::memset(&gp, 0, sizeof gp);
    fill_generic_specs(e, gp);
    if (e->words < 1 || e->words > 24) return BGR_OK;  // the row has to fit the register file
    for (uint32_t c = 0; c < gp.n_hash; ++c)   // whole-word byte ranges only (every POD of u32 / f32 / u64 fields)
        if (((gp.hash[c].off | gp.hash[c].len) & 3u) != 0u || gp.hash[c].len < 4 || gp.hash[c].len > 64)
            return user ? fail(BGR_ERR_UNSUPPORTED, "user systems need every checksummed byte range to be 4..64 whole words") : BGR_OK;
    const std::string user_pre = user ? user_systems_prelude(e) : std::string();
    const int rows = e->tune_jit_rows == 1 || e->tune_jit_rows == 2 ? e->tune_jit_rows : 4;
    int rc = BGR_OK;
    auto compile = [&](int item_rows, int rows, JitKernel* out) {
        const int threads = item_rows / rows;
        std::string pre;
        auto def = [&](const char* name, unsigned long long v) { pre += "#define " + std::string(name) + " " + std::to_string(v) + "\n"; };
        def("BGR_SYS_PARTICLES_UPDATE", BGR_SYS_PARTICLES_UPDATE); def("BGR_SYS_PARTICLES_DESPAWN", BGR_SYS_PARTICLES_DESPAWN);
        def("BGR_SYS_BOX_MOVE", BGR_SYS_BOX_MOVE); def("BGR_SYS_U32_ADD", BGR_SYS_U32_ADD);
        def("BGR_SYS_U32_SATSUB_DESPAWN", BGR_SYS_U32_SATSUB_DESPAWN); def("BGR_SYS_U32_STORE_CALL_COUNT", BGR_SYS_U32_STORE_CALL_COUNT);
        def("BGR_SYS_PARTICLES_SPAWN", BGR_SYS_PARTICLES_SPAWN); def("BGR_SYS_DESPAWN_ON_INPUT", BGR_SYS_DESPAWN_ON_INPUT);
        def("BGR_TILE_ROWS", kTileRows);
        def("BGR_JIT_WORDS", e->words); def("BGR_JIT_ROWS", rows); def("BGR_JIT_ITEM_ROWS", item_rows);
        // resident blocks the register allocation has to allow: ~512 threads per SM for narrow rows, ~256 for wide ones
        def("BGR_JIT_MINB", std::max(1, (e->words <= 8 ? 512 : 256) / threads));
        def("BGR_JIT_NSYS", gp.n_sys); def("BGR_JIT_NHASH", gp.n_hash);
        auto u = [](uint32_t v) { return std::to_string(v) + "u"; };
        pre += "#define BGR_JIT_SYS_LIST ";
        for (uint32_t i = 0; i < gp.n_sys; ++i) {
            const SysSpec& y = gp.sys[i];
            pre += "{" + u(y.id) + "," + u(y.plane0) + "," + u(y.plane1) + "," + u(y.need) + "," + u(y.param) + "}, ";
        }
        pre += "{0u,0u,0u,0u,0u}\n#define BGR_JIT_HASH_LIST ";
        for (uint32_t i = 0; i < gp.n_hash; ++i) {
            const HashSpec& h = gp.hash[i];
            pre += "{" + u(h.first_plane) + "," + u(h.off) + "," + u(h.len) + "," + u(h.finite) + "," + u(h.slot) + "," + u(h.absent) + "}, ";
        }
        pre += "{0u,0u,0u,0u,0u,0u}\n";
        pre += user_pre;
        std::string why;
        bool compile_error = false;
        const bool ok = jit_generic_program(pre, threads, reinterpret_cast<const void*>(&bgr_abi_version), out, &why, &compile_error);
        if (!ok && user && rc == BGR_OK)
            rc = fail(compile_error ? BGR_ERR_INVALID_ARGUMENT : BGR_ERR_UNSUPPORTED, "user systems cannot be compiled: " + why);
        else if (!ok && std::getenv("BGR_JIT_VERBOSE"))
            std::fprintf(stderr, "[bevy_ggrs_b200] generic program not specialised, the interpreter kernel runs: %s\n", why.c_str());
        out->item_rows = item_rows;
    };
    const int forced = e->tune_jit_item == 512 || e->tune_jit_item == 256 || e->tune_jit_item == 128 ? e->tune_jit_item : 0;
    compile(forced ? forced : int(kTileRows), std::min(rows, (forced ? forced : int(kTileRows)) / 32), &e->jit);  // a block is at least one warp
    // worlds of few tiles per SM: quarter-tile items, two rows per thread (measured: profiles/r02_generic_jit_sweep.txt)
    if (!forced && e->jit.fn) compile(128, 2, &e->jit_small);
    if (rc != BGR_OK) { e->jit = JitKernel{}; e->jit_small = JitKernel{}; }
    return rc;
}

// ---------------------------------------------------------------------------------------------
// launch: generic one-launch program (any schema, compiled systems; generic_program.cuh)
// ---------------------------------------------------------------------------------------------
int run_generic(bgr_engine* e, const Program& pg, uint32_t buf) {
    e->main_dirty = true;
    const bool prev_chain = e->tiledep_chain;  // the last operation on the stream was a signalling launch of the generated kernel
    e->tiledep_chain = false;
    GenericParams gp;
    std::memset(&gp, 0, sizeof gp);
    gp.arena = e->arena;
    gp.order_base = e->cfg.order_base;
    gp.accum = e->d_accum_c[0];
    gp.ticket = e->d_ticket_c[0];
    gp.out = e->d_out[buf];
    gp.seq = e->seq;
    if (e->d_trace && e->seq - e->trace_first_seq < e->trace_cap) gp.trace = e->d_trace + (e->seq - e->trace_first_seq) * 4;
    gp.words = e->words; gp.tile_bytes = e->tile_bytes;
    gp.n_ops = pg.n_ops; gp.n_saves = pg.n_saves;
    gp.n_tiles = std::max(1u, e->tiles_for(pg.max_rows));
    gp.live_rows = pg.live_rows;
    if (!pg.first_is_load) gp.flags |= PF_READ_LIVE;
    if (pg.has_load || pg.has_advance) gp.flags |= PF_WRITE_LIVE_ACTIVE;
    fill_generic_specs(e, gp);
    std::memcpy(gp.ops, pg.ops, sizeof(Op) * pg.n_ops);
    std::memcpy(gp.adv_frame, pg.adv_frame, sizeof(int32_t) * pg.n_ops);
    if (e->jit.fn) {  // the registration's own register-resident kernel
        // few tiles per SM: with whole tiles some SMs carry twice the rows of others and set the kernel's duration
        const JitKernel& k = (e->jit_small.fn && gp.n_tiles < 3u * uint32_t(e->num_sms)) ? e->jit_small : e->jit;
        const uint32_t n_items = gp.n_tiles * (kTileRows / uint32_t(k.item_rows));
        uint32_t grid = std::max(1u, std::min(n_items, uint32_t(e->num_sms * k.bps)));
        if (e->tune_grid > 0) grid = std::min(grid, uint32_t(e->tune_grid));
        // Overlap of consecutive launches: only when request vectors are queued behind each other (a synchronous caller
        // collects before its next submit), only on a stream the engine owns, and only between launches of the SAME kernel
        // over the SAME items (the per-item flags mean nothing across partitions: drain instead — rare, rows crossed a tile).
        const bool tiledep = e->tune_jit_tiledep && e->d_item_done && e->own_stream && (e->tune_jit_tiledep > 1 || !e->pending.empty());
        bool wait = false;
        if (prev_chain) {
            if (tiledep && e->jit_chain_kernel == k.fn && e->tiledep_tiles == n_items) wait = true;
            else CUDA_TRY(cudaStreamSynchronize(e->stream));  // an earlier overlapping launch may still be running
        }
        if (tiledep) {
            gp.flags |= PF_TILE_SIGNAL;
            gp.item_done = e->d_item_done;
            gp.done_seq = uint32_t(e->seq);
            if (wait) { gp.flags |= PF_TILE_WAIT; gp.wait_seq = e->tiledep_seq; gp.wait_items = n_items; }
            // overlapping launches must not share accumulators / tickets: one set per in-flight request vector (run_fused)
            const uint32_t set = uint32_t(e->seq % bgr_engine::kBufs);
            gp.accum = e->d_accum_c[set];
            gp.ticket = e->d_ticket_c[set];
        }
        void* args[] = {&gp};
        cudaLaunchConfig_t cfg;
        std::memset(&cfg, 0, sizeof cfg);
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(k.threads); cfg.dynamicSmemBytes = 0; cfg.stream = e->stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = wait ? 1u : 0u;
        CUDA_TRY(cudaLaunchKernelExC(&cfg, k.fn, args));
        CUDA_TRY(cudaGetLastError());
        e->launches += 1;
        e->tiledep_chain = tiledep;
        e->tiledep_seq = uint32_t(e->seq); e->tiledep_tiles = n_items; e->jit_chain_kernel = k.fn;
        return BGR_OK;
    }
    const size_t smem = size_t((e->tile_bytes + 127u) & ~127u);
    // rows of a tile per thread: 8 (64 threads per tile), 4 (128), 2 (256) or 1 (512).  More rows per thread = more
    // independent hash chains interleaved in one warp; measured (scripts/gpu_generic_block.sh): see DESIGN.md
    const int block = e->tune_generic_block == 64 || e->tune_generic_block == 256 || e->tune_generic_block == 512 ? e->tune_generic_block : 128;
    const int vi = block == 64 ? 0 : block == 128 ? 1 : block == 256 ? 2 : 3;
    const void* fn = vi == 0 ? (const void*)k_generic_program<64> : vi == 1 ? (const void*)k_generic_program<128>
                   : vi == 2 ? (const void*)k_generic_program<256> : (const void*)k_generic_program<512>;
    if (e->generic_bps[vi] == 0) {
        if (smem > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
        int nb = 0;
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, block, smem));
        e->generic_bps[vi] = std::max(1, nb);
    }
    uint32_t grid = std::max(1u, std::min(gp.n_tiles, uint32_t(e->num_sms * e->generic_bps[vi])));
    if (e->tune_grid > 0) grid = std::min(grid, uint32_t(e->tune_grid));  // tests: several tiles per block on small worlds
    void* args[] = {&gp};
    CUDA_TRY(cudaLaunchKernel(fn, dim3(grid), dim3(block), args, smem, e->stream));
    CUDA_TRY(cudaGetLastError());
    e->launches += 1;
    return BGR_OK;
}


int submit(bgr_engine* e, const bgr_session_info* sess, const bgr_request* reqs, uint32_t n) {
    NvtxRange span("HandleRequests");
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    if (!e->built) return fail(BGR_ERR_STATE, "bgr_build has not been called");
    if (e->pending.size() >= size_t(bgr_engine::kBufs)) return fail(BGR_ERR_STATE, "too many un-collected submits");
    if (n && !reqs) return fail(BGR_ERR_INVALID_ARGUMENT, "null requests");
    const uint64_t t_begin = host_ns();
    HostState s = e->st;
    Program pg;
    int rc = compile_requests(e, s, sess, reqs, n, pg);
    if (rc != BGR_OK) return rc;  // nothing executed, nothing committed
    const uint64_t t_compiled = host_ns();
    uint32_t buf = e->next_buf;
    if (e->group) {
        // the buffer of this request vector was last used kBufs vectors ago: every peer must have folded that one
        std::string err;
        if (!e->group->wait_reusable(e->gseq + 1, &err)) return fail(BGR_ERR_STATE, err);
        e->gseq += 1;
        buf = ShardGroup::buf_of(e->gseq);
        e->group->publish_meta(e->gseq, pg.n_saves, e->n_ck, pg.save_frames, pg.save_totals);
    }
    if (!pg.spawn_vals.empty()) std::memcpy(e->h_spawn[buf], pg.spawn_vals.data(), pg.spawn_vals.size() * sizeof(float2));
    e->seq += 1;
    e->ticked = true;
    const bool stepwise_forced = e->cfg.flags & BGR_CFG_FORCE_STEPWISE;
    const bool bundle = e->bundle_particles && e->tune_bundle && !stepwise_forced;
    const bool generic = !bundle && e->generic_ok && e->tune_generic && !stepwise_forced;
    const bool fused = bundle || generic;   // one launch for the whole request vector
    uint32_t chains = 1;
    rc = bundle ? run_fused(e, pg, buf, &chains) : generic ? run_generic(e, pg, buf) : run_stepwise(e, pg, buf);
    if (rc != BGR_OK) return rc;
    // an event between two launches would serialise them; with host polling it is only a fallback, taken lazily
    if (!(e->tune_tiledep && e->tune_poll)) CUDA_TRY(cudaEventRecord(e->ev[buf], e->stream));
    e->last_fused = fused;
    e->st = s;
    Pending pd;
    pd.buf = buf; pd.n_saves = pg.n_saves; pd.seq = e->seq; pd.chains = chains; pd.gseq = e->group ? e->gseq : 0;
    std::memcpy(pd.frames, pg.save_frames, sizeof(int32_t) * pg.n_saves);
    std::memcpy(pd.totals, pg.save_totals, sizeof(uint32_t) * pg.n_saves);
    e->pending.push_back(pd);
    e->next_buf = (buf + 1) % bgr_engine::kBufs;
    e->prof[0] += 1; e->prof[1] += t_compiled - t_begin; e->prof[2] += host_ns() - t_compiled;
    return BGR_OK;
}

void fold(const bgr_partial& p, bgr_checksum* out) {
    // EntityChecksumPlugin::update (entity_checksum.rs:35-43)
    uint64_t x = sea_hash_2xu64(p.active, p.total);
    // ComponentChecksumPlugin: `result.hash(&mut hasher)` (component_checksum.rs:93-95), then
    // ChecksumPlugin::update XORs every part (checksum.rs:88-99)
    for (uint32_t c = 0; c < p.n_columns && c < BGR_MAX_CHECKSUM_COLUMNS; ++c) x ^= sea_hash_u64(p.xor_[c]);
    out->frame = p.frame;
    out->has_checksum = 1;
    out->lo = x;
    out->hi = 0;
}

int collect(bgr_engine* e, bgr_checksum* out, uint32_t cap, uint32_t* n_out) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    if (e->pending.empty()) return fail(BGR_ERR_STATE, "nothing to collect");
    Pending pd = e->pending.front();
    e->pending.pop_front();
    const uint64_t t_wait0 = host_ns();
    // Completion: the last block of each chain's kernel publishes every result word as a self-validating pair
    // (v, v ^ result_tag(seq, i)) plus a completion pair; a word is accepted when its halves XOR to this launch's tag.
    unsigned long long folded[kMaxSaves * kAccStride];
    for (uint32_t i = 0; i < pd.n_saves * kAccStride; ++i) folded[i] = 0;
    const uint32_t n_words = pd.n_saves * kAccStride;
    for (uint32_t c = 0; c < pd.chains; ++c) {
        const volatile unsigned long long* blk = &e->h_out[pd.buf][size_t(c) * kResultStride];
        unsigned long long words[kMaxSaves * kAccStride];
        uint32_t valid = 0;
        bool seq_ok = false;
        auto ready = [&]() {
            if (!seq_ok) {
                const unsigned long long a = blk[2 * kSeqIndex], b = blk[2 * kSeqIndex + 1];
                if ((a ^ b) != result_tag(pd.seq, kSeqIndex)) return false;
                seq_ok = true;
            }
            while (valid < n_words) {
                const unsigned long long a = blk[2 * valid], b = blk[2 * valid + 1];
                if ((a ^ b) != result_tag(pd.seq, valid)) return false;
                words[valid++] = a;
            }
            return true;
        };
        bool done = false;
        if (e->tune_poll && !pd.finished) {
            for (int spin = 0; spin < 200000; ++spin) {
                if (ready()) { done = true; break; }
                __builtin_ia32_pause();
            }
        }
        if (!done) {  // the event / the stream is ordered after every chain
            if (!pd.finished) {
                if (e->tune_tiledep && e->tune_poll) CUDA_TRY(cudaStreamSynchronize(e->stream));
                else CUDA_TRY(cudaEventSynchronize(e->ev[pd.buf]));
            }
            if (!ready()) return fail(BGR_ERR_CUDA, "request vector completed without publishing valid results");
        }
        // fold the chains' result blocks: XOR the column words, sum the live-row counts, OR the flags
        for (uint32_t i = 0; i < n_words; ++i) {
            const uint32_t w = i % kAccStride;
            if (w == 6) folded[i] += words[i]; else if (w == 7) folded[i] |= words[i]; else folded[i] ^= words[i];
        }
    }
    const uint64_t t_wait1 = host_ns();
    e->prof[3] += t_wait1 - t_wait0;
    const unsigned long long* r = folded;
    e->last_partials.clear();
    bool nonfinite = false;
    // shard group: wait for every rank's block of this request vector and combine (XOR / sum / OR) across ranks
    bgr_partial combined[kMaxSaves];
    if (pd.gseq) {
        uint32_t n = 0;
        uint64_t flags = 0;
        std::string err;
        if (!e->group || !e->group->combine(pd.gseq, combined, kMaxSaves, &n, &flags, &err))
            return fail(BGR_ERR_STATE, e->group ? err : "request vector was submitted inside a shard group that has been left");
        if (flags & 1ULL) nonfinite = true;
    }
    for (uint32_t k = 0; k < pd.n_saves; ++k) {
        bgr_partial p;
        std::memset(&p, 0, sizeof p);
        p.frame = pd.frames[k];
        p.n_columns = e->n_ck;
        p.active = r[k * kAccStride + 6];
        p.total = pd.totals[k];
        for (uint32_t c = 0; c < e->n_ck; ++c) p.xor_[c] = r[k * kAccStride + c];
        if (r[k * kAccStride + 7] & 1ULL) nonfinite = true;
        e->last_partials.push_back(p);
    }
    if (n_out) *n_out = pd.n_saves;
    for (uint32_t k = 0; k < pd.n_saves && k < cap && out; ++k) {
        if (pd.gseq) {
            fold(combined[k], &out[k]);  // the frame checksum of the WHOLE world, identical on every rank
        } else if (e->cfg.flags & BGR_CFG_SHARDED) {
            out[k].frame = pd.frames[k]; out[k].has_checksum = 0; out[k].lo = 0; out[k].hi = 0;
        } else {
            fold(e->last_partials[k], &out[k]);
        }
    }
    e->prof[4] += host_ns() - t_wait1;
    if (nonfinite) return fail(BGR_ERR_NON_FINITE, "Hashing is not stable for NaN f32 values.");
    return BGR_OK;
}

// Entry points that touch the live world (read / write / spawn / peek ...) first wait for every submitted request
// vector.  The results of un-collected submits STAY queued: a later bgr_collect still returns their checksums (and
// the non-finite status), in order — nothing is dropped on the floor.
int drain(bgr_engine* e) {
    e->tiledep_chain = false;  // callers enqueue ordinary (fully ordered) work next
    if (e->pending.empty()) return BGR_OK;
    CUDA_TRY(cudaStreamSynchronize(e->stream));  // every chain stream is joined into the main stream by an event
    e->pending.for_each([](Pending& pd) { pd.finished = true; });
    return BGR_OK;
}

int ensure_stage(bgr_engine* e, size_t bytes) {
    if (bytes <= e->stage_cap) return BGR_OK;
    if (e->d_stage) CUDA_TRY(cudaFree(e->d_stage));
    e->d_stage = nullptr; e->stage_cap = 0;
    size_t cap = std::max<size_t>(bytes, 1u << 20);
    CUDA_TRY(cudaMalloc(&e->d_stage, cap));
    e->stage_cap = cap;
    return BGR_OK;
}

// ECS column (array of T, `stride` bytes apart) <-> tile-planar image: one H2D/D2H copy of the AoS
// bytes + one transposition kernel (k_scatter_column / k_gather_column).
int transfer_column(bgr_engine* e, uint32_t image_idx, uint32_t column, uint32_t first, uint32_t count, void* host,
                    uint32_t stride, bool to_device) {
    if (!e || !e->built) return fail(BGR_ERR_STATE, "engine not built");
    if (column >= e->cols.size()) return fail(BGR_ERR_INVALID_ARGUMENT, "unknown column");
    const Column& c = e->cols[column];
    if (stride < c.elem_bytes) return fail(BGR_ERR_INVALID_ARGUMENT, "stride < elem_bytes");
    if (uint64_t(first) + count > e->cfg.max_entities) return fail(BGR_ERR_CAPACITY, "row range exceeds max_entities");
    if (count == 0) return BGR_OK;
    int rc = drain(e);
    if (rc != BGR_OK) return rc;
    const size_t bytes = size_t(count) * stride;
    rc = ensure_stage(e, bytes);
    if (rc != BGR_OK) return rc;
    uint8_t* img = e->image(image_idx);
    uint32_t grid = e->grid_for(uint32_t(std::min<size_t>(size_t(count) * c.words, 0x7fffffffu)), 256);
    if (to_device) {
        e->st.live_passive_ver = ++e->st.ver_counter;  // host wrote a column: live content is new
        CUDA_TRY(cudaMemcpyAsync(e->d_stage, host, bytes, cudaMemcpyHostToDevice, e->stream));
        k_scatter_column<<<grid, 256, 0, e->stream>>>(img, e->words, c.first_plane, c.words, c.elem_bytes, first, count, e->d_stage, stride);
        e->launches += 1;
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaStreamSynchronize(e->stream));
    } else {
        if (stride != c.elem_bytes) CUDA_TRY(cudaMemcpyAsync(e->d_stage, host, bytes, cudaMemcpyHostToDevice, e->stream));  // keep the caller's padding bytes
        k_gather_column<<<grid, 256, 0, e->stream>>>(img, e->words, c.first_plane, c.words, c.elem_bytes, first, count, e->d_stage, stride);
        e->launches += 1;
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemcpyAsync(host, e->d_stage, bytes, cudaMemcpyDeviceToHost, e->stream));
        CUDA_TRY(cudaStreamSynchronize(e->stream));
    }
    return BGR_OK;
}

int read_alive_image(bgr_engine* e, uint32_t image_idx, uint32_t first, uint32_t count, uint32_t n_rows, uint8_t* dst,
                     uint32_t need = 0) {
    if (count == 0) return BGR_OK;
    int rc = drain(e);
    if (rc != BGR_OK) return rc;
    if (uint64_t(first) + count > e->cfg.max_entities) return fail(BGR_ERR_CAPACITY, "row range exceeds max_entities");
    rc = ensure_stage(e, count);
    if (rc != BGR_OK) return rc;
    k_gather_alive<<<e->grid_for(count, 256), 256, 0, e->stream>>>(e->image(image_idx), e->words, first, count, n_rows, e->d_stage, need);
    e->launches += 1;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(dst, e->d_stage, count, cudaMemcpyDeviceToHost, e->stream));
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    return BGR_OK;
}

int download_begin(bgr_engine* e, uint32_t column, uint32_t off, uint32_t len, uint32_t first, uint32_t count, void* host,
                   uint32_t* ticket_out) {
    if (!e || !e->built) return fail(BGR_ERR_STATE, "engine not built");
    if (!host || !ticket_out) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    if (column >= e->cols.size()) return fail(BGR_ERR_INVALID_ARGUMENT, "unknown column");
    const Column& c = e->cols[column];
    if ((off & 3u) || (len & 3u) || len == 0 || uint64_t(off) + len > uint64_t(c.words) * 4u)
        return fail(BGR_ERR_INVALID_ARGUMENT, "field range must be 4-byte aligned and inside the element");
    if (uint64_t(first) + count > e->st.n_rows) return fail(BGR_ERR_CAPACITY, "row range exceeds the spawned rows");
    uint32_t slot = BGR_MAX_DOWNLOADS;
    for (uint32_t k = 0; k < BGR_MAX_DOWNLOADS; ++k) {
        const uint32_t i = (e->next_dl + k) % BGR_MAX_DOWNLOADS;
        if (!e->dl[i].busy) { slot = i; break; }
    }
    if (slot == BGR_MAX_DOWNLOADS) return fail(BGR_ERR_STATE, "too many downloads in flight (BGR_MAX_DOWNLOADS)");
    bgr_engine::Download& d = e->dl[slot];
    const size_t bytes = size_t(count) * len;
    if (!e->copy_stream) CUDA_TRY(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
    if (!d.packed) {
        CUDA_TRY(cudaEventCreateWithFlags(&d.packed, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&d.done, cudaEventDisableTiming));
    }
    if (bytes > d.cap) {  // grows to the largest request and stays (the slot is idle: its last copy was waited for)
        if (d.d_buf) CUDA_TRY(cudaFree(d.d_buf));
        d.d_buf = nullptr; d.cap = 0;
        CUDA_TRY(cudaMalloc(&d.d_buf, bytes));
        d.cap = bytes;
    }
    if (count) {
        const uint32_t n_words = len / 4u;
        const uint32_t grid = e->grid_for(uint32_t(std::min<size_t>(size_t(count) * n_words, 0x7fffffffu)), 256);
        k_gather_fields<<<grid, 256, 0, e->stream>>>(e->image(0), e->words, c.first_plane + off / 4u, n_words, first, count,
                                                      reinterpret_cast<uint32_t*>(d.d_buf));
        e->launches += 1;
        CUDA_TRY(cudaGetLastError());
        e->main_dirty = true;  // later chain launches overwrite the live image this kernel reads
        e->tiledep_chain = false;
        CUDA_TRY(cudaEventRecord(d.packed, e->stream));
        CUDA_TRY(cudaStreamWaitEvent(e->copy_stream, d.packed, 0));
        CUDA_TRY(cudaMemcpyAsync(host, d.d_buf, bytes, cudaMemcpyDeviceToHost, e->copy_stream));
    }
    CUDA_TRY(cudaEventRecord(d.done, e->copy_stream));
    d.busy = true;
    e->next_dl = (slot + 1) % BGR_MAX_DOWNLOADS;
    *ticket_out = slot;
    return BGR_OK;
}

int download_wait(bgr_engine* e, uint32_t ticket) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    if (ticket >= BGR_MAX_DOWNLOADS || !e->dl[ticket].busy) return fail(BGR_ERR_STATE, "no such download in flight");
    CUDA_TRY(cudaEventSynchronize(e->dl[ticket].done));
    e->dl[ticket].busy = false;
    return BGR_OK;
}

void detect_bundles(bgr_engine* e) {
    e->bundle_particles = false;
    e->passive.clear();
    e->bundle_opt = false;
    for (const Column& c : e->cols)
        if (c.absent) e->bundle_opt = true;  // per-entity presence: the MODE 2 variant of the fused kernel
    const SystemReg* up = nullptr; const SystemReg* de = nullptr; const SystemReg* sp = nullptr;
    for (auto& s : e->systems) {
        if (s.id == BGR_SYS_PARTICLES_UPDATE && !up) up = &s;
        else if (s.id == BGR_SYS_PARTICLES_DESPAWN && !de) de = &s;
        else if (s.id == BGR_SYS_PARTICLES_SPAWN && !sp) sp = &s;
        else return;  // any other system: generic path
    }
    if (!up || !de) return;
    uint32_t t = up->cols[0], v = up->cols[1], l = de->cols[0];
    if (sp && (sp->cols[0] != t || sp->cols[1] != v || sp->cols[2] != l)) return;
    if (t == v || t == l || v == l) return;
    auto ck_ok = [&](const Column& c) {
        return c.hash_kind == BGR_HASH_NONE || (c.hash_kind == BGR_HASH_BYTES && c.hash_off == 0 && c.hash_len == 12);
    };
    if (!ck_ok(e->cols[t]) || !ck_ok(e->cols[v])) return;
    for (size_t i = 0; i < e->cols.size(); ++i)
        if (i != t && i != v && e->cols[i].hash_kind != BGR_HASH_NONE) return;  // other checksums: generic path
    // active planes: translation (3 words of Transform), velocity (3), ttl (2)
    std::vector<uint8_t> active(e->words, 0);
    for (uint32_t k = 0; k < 3; ++k) { active[e->cols[t].first_plane + k] = 1; active[e->cols[v].first_plane + k] = 1; }
    for (uint32_t k = 0; k < 2; ++k) active[e->cols[l].first_plane + k] = 1;
    for (uint32_t p = 0; p < e->words; ++p)
        if (!active[p]) e->passive.push_back(uint16_t(p));
    if (e->passive.size() > size_t(kMaxPassive)) { e->passive.clear(); return; }
    // runs of adjacent passive planes: one cp.async.bulk each
    e->runs.clear(); e->passive_bytes = 0;
    for (size_t i = 0; i < e->passive.size();) {
        size_t j = i;
        while (j + 1 < e->passive.size() && e->passive[j + 1] == e->passive[j] + 1) ++j;
        PassiveRun r{uint32_t(e->passive[i]) * kPlaneBytes, uint32_t(j - i + 1) * kPlaneBytes};
        e->runs.push_back(r);
        e->passive_bytes += r.bytes;
        i = j + 1;
    }
    if (e->runs.size() > size_t(kMaxRuns)) { e->runs.clear(); e->passive_bytes = 0; }
    const bool fin_t = e->cols[t].hash_flags & BGR_HASH_FLAG_ASSERT_FINITE_F32, fin_v = e->cols[v].hash_flags & BGR_HASH_FLAG_ASSERT_FINITE_F32;
    const bool ck_t = e->cols[t].hash_kind != BGR_HASH_NONE, ck_v = e->cols[v].hash_kind != BGR_HASH_NONE;
    e->bundle_static_ck = ck_t && ck_v && fin_t && fin_v;
    e->bt = t; e->bv = v; e->bl = l;
    e->bundle_particles = true;
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

BGR_API uint32_t bgr_abi_version(void) { return BGR_ABI_VERSION; }
BGR_API const char* bgr_last_error(void) { return g_err.c_str(); }

BGR_API int bgr_engine_create(const bgr_config* cfg, bgr_engine** out) {
    if (!cfg || !out) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    if (cfg->abi_version != BGR_ABI_VERSION) return fail(BGR_ERR_INVALID_ARGUMENT, "ABI version mismatch");
    if (cfg->max_entities == 0 || cfg->fps == 0) return fail(BGR_ERR_INVALID_ARGUMENT, "max_entities and fps must be > 0");
    if (cfg->max_depth == 0 || cfg->max_depth > 64) return fail(BGR_ERR_INVALID_ARGUMENT, "max_depth must be in 1..64");
    int n_dev = 0;
    cudaError_t ce = cudaGetDeviceCount(&n_dev);
    if (ce != cudaSuccess || n_dev == 0)
        return fail(BGR_ERR_CUDA, std::string("no CUDA device available (bevy_ggrs_b200 has no CPU fallback): ") + cudaGetErrorString(ce));
    if (cfg->device < 0 || cfg->device >= n_dev) return fail(BGR_ERR_INVALID_ARGUMENT, "bad device ordinal");
    CUDA_TRY(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major < 10)
        return fail(BGR_ERR_CUDA, "device is not sm_100 (Blackwell); this library only carries sm_100a code");
    bgr_engine* e = new bgr_engine();
    e->cfg = *cfg;
    e->num_sms = prop.multiProcessorCount;
    if (cfg->stream) { e->stream = static_cast<cudaStream_t>(cfg->stream); e->own_stream = false; }
    else {
        cudaError_t se = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking);
        if (se != cudaSuccess) { delete e; return fail(BGR_ERR_CUDA, cudaGetErrorString(se)); }
        e->own_stream = true;
    }
    e->tune_vec = env_int("BGR_TUNE_VEC", 2);
    e->tune_minb = env_int("BGR_TUNE_MINB", 2);
    e->tune_bps = env_int("BGR_TUNE_BPS", 0);
    e->tune_tma = env_int("BGR_TUNE_TMA", 1);
    e->tune_passive_tma = env_int("BGR_TUNE_PASSIVE_TMA", 1);
    e->tune_poll = env_int("BGR_TUNE_POLL", 1);
    e->tune_dynamic = env_int("BGR_TUNE_DYNAMIC", 1);
    e->tune_pdl = env_int("BGR_TUNE_PDL", 0);
    e->tune_prefetch = env_int("BGR_TUNE_PREFETCH", 1);
    e->tune_grid = env_int("BGR_TUNE_GRID", 0);
    e->tune_tiledep = env_int("BGR_TUNE_TILEDEP", 1);
    e->tune_generic = env_int("BGR_TUNE_GENERIC", 1);
    e->tune_sub = env_int("BGR_TUNE_SUB", 0);
    e->tune_generic_block = env_int("BGR_TUNE_GENERIC_BLOCK", 0);
    e->tune_jit = env_int("BGR_TUNE_JIT", 1);
    e->tune_jit_rows = env_int("BGR_TUNE_JIT_ROWS", 4);
    e->tune_jit_item = env_int("BGR_TUNE_JIT_ITEM", 0);
    e->tune_jit_tiledep = env_int("BGR_TUNE_JIT_TILEDEP", 0);
    e->tune_passive_early = env_int("BGR_TUNE_PASSIVE_EARLY", -1);
    e->tune_stagger_ns = env_int("BGR_TUNE_STAGGER_NS", 800);
    e->tune_bundle = env_int("BGR_TUNE_BUNDLE", 1);
    e->n_chains = std::max(1, std::min(int(bgr_engine::kMaxChains), env_int("BGR_TUNE_CHAINS", 1)));
    if (e->tune_vec != 1 && e->tune_vec != 2 && e->tune_vec != 4) e->tune_vec = 2;
    e->st.confirmed = 0;
    *out = e;
    return BGR_OK;
}

BGR_API void bgr_engine_destroy(bgr_engine* e) {
    if (!e) return;
    cudaSetDevice(e->cfg.device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    if (e->group) {
        cudaHostUnregister(e->group->blocks_base());
        for (int b = 0; b < bgr_engine::kBufs; ++b) { e->h_out[b] = e->own_h_out[b]; e->d_out[b] = e->own_d_out[b]; }
        delete e->group;
        e->group = nullptr;
    }
    if (e->d_trace) cudaFree(e->d_trace);
    for (int i = 0; i < bgr_engine::kBufs; ++i) {
        if (e->h_out[i]) cudaFreeHost(e->h_out[i]);
        if (e->h_spawn[i]) cudaFreeHost(e->h_spawn[i]);
        if (e->ev[i]) cudaEventDestroy(e->ev[i]);
    }
    if (e->arena) cudaFree(e->arena);
    if (e->d_kill) cudaFree(e->d_kill);
    if (e->d_stage) cudaFree(e->d_stage);
    if (e->d_accum) cudaFree(e->d_accum);
    if (e->d_ticket) cudaFree(e->d_ticket);
    if (e->copy_stream) { cudaStreamSynchronize(e->copy_stream); cudaStreamDestroy(e->copy_stream); }
    if (e->d_tma_ticket) cudaFree(e->d_tma_ticket);
    if (e->d_tile_done) cudaFree(e->d_tile_done);
    if (e->d_tile_cnt) cudaFree(e->d_tile_cnt);
    if (e->d_item_done) cudaFree(e->d_item_done);
    for (auto& d : e->dl) {
        if (d.d_buf) cudaFree(d.d_buf);
        if (d.packed) cudaEventDestroy(d.packed);
        if (d.done) cudaEventDestroy(d.done);
    }
    for (int c = 0; c < bgr_engine::kMaxChains; ++c) {
        if (e->chain_stream[c]) { cudaStreamSynchronize(e->chain_stream[c]); cudaStreamDestroy(e->chain_stream[c]); }
        if (e->chain_ev[c]) cudaEventDestroy(e->chain_ev[c]);
    }
    if (e->main_ev) cudaEventDestroy(e->main_ev);
    if (e->own_stream && e->stream) cudaStreamDestroy(e->stream);
    delete e;
}

BGR_API int bgr_rollback_component(bgr_engine* e, const char* type_name, uint32_t elem_bytes, uint32_t strategy,
                                   uint32_t* column_out) {
    if (!e || !column_out) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    if (e->built) return fail(BGR_ERR_STATE, "components must be registered before bgr_build");
    if (elem_bytes == 0 || elem_bytes > 1024) return fail(BGR_ERR_INVALID_ARGUMENT, "elem_bytes must be in 1..1024");
    const bool optional = strategy & BGR_STRATEGY_OPTIONAL;
    strategy &= ~BGR_STRATEGY_OPTIONAL;
    if (strategy != BGR_STRATEGY_COPY && strategy != BGR_STRATEGY_CLONE)
        return fail(BGR_ERR_UNSUPPORTED, "only Copy/Clone strategies of POD types are supported (ReflectStrategy is out of scope)");
    Column c;
    if (optional) {
        uint32_t n_opt = 0;
        for (const Column& o : e->cols) n_opt += o.absent ? 1u : 0u;
        if (n_opt >= BGR_MAX_OPTIONAL_COLUMNS) return fail(BGR_ERR_CAPACITY, "more than BGR_MAX_OPTIONAL_COLUMNS optional columns");
        c.absent = 2u << n_opt;
    }
    c.name = type_name ? type_name : "";
    c.elem_bytes = elem_bytes;
    c.words = (elem_bytes + 3) / 4;
    c.strategy = strategy;
    e->cols.push_back(c);
    *column_out = uint32_t(e->cols.size() - 1);
    return BGR_OK;
}

BGR_API int bgr_checksum_component(bgr_engine* e, uint32_t column, uint32_t hash_kind, uint32_t byte_offset,
                                   uint32_t byte_len, uint32_t flags) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    if (e->built) return fail(BGR_ERR_STATE, "checksums must be registered before bgr_build");
    if (column >= e->cols.size()) return fail(BGR_ERR_INVALID_ARGUMENT, "unknown column");
    Column& c = e->cols[column];
    if (hash_kind != BGR_HASH_BYTES) return fail(BGR_ERR_INVALID_ARGUMENT, "unknown hash kind");
    if (uint64_t(byte_offset) + byte_len > c.elem_bytes) return fail(BGR_ERR_INVALID_ARGUMENT, "hash range exceeds element");
    if ((flags & BGR_HASH_FLAG_ASSERT_FINITE_F32) && ((byte_offset | byte_len) & 3u))
        return fail(BGR_ERR_INVALID_ARGUMENT, "finite-f32 assertion needs a 4-byte aligned range");
    c.hash_kind = hash_kind; c.hash_off = byte_offset; c.hash_len = byte_len; c.hash_flags = flags;
    return BGR_OK;
}

BGR_API int bgr_add_system(bgr_engine* e, uint32_t system, const uint32_t* columns, uint32_t n_columns,
                           const uint32_t* params, uint32_t n_params) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    if (e->built) return fail(BGR_ERR_STATE, "systems must be added before bgr_build");
    SystemReg s;
    s.id = system;
    for (uint32_t i = 0; i < n_columns; ++i) {
        if (columns[i] >= e->cols.size()) return fail(BGR_ERR_INVALID_ARGUMENT, "system binds an unknown column");
        s.cols.push_back(columns[i]);
    }
    for (uint32_t i = 0; i < n_params; ++i) s.params.push_back(params[i]);
    auto need = [&](size_t nc, size_t np) { return s.cols.size() == nc && s.params.size() >= np; };
    auto eb = [&](size_t i) { return e->cols[s.cols[i]].elem_bytes; };
    switch (system) {
    case BGR_SYS_PARTICLES_UPDATE:
        if (!need(2, 0) || eb(0) != 40 || eb(1) != 12)
            return fail(BGR_ERR_INVALID_ARGUMENT, "update_particles binds {Transform(40B), Velocity(12B)}");
        break;
    case BGR_SYS_PARTICLES_DESPAWN:
        if (!need(1, 0) || eb(0) != 8) return fail(BGR_ERR_INVALID_ARGUMENT, "despawn_particles binds {Ttl(8B)}");
        break;
    case BGR_SYS_U32_ADD:
    case BGR_SYS_U32_SATSUB_DESPAWN:
        if (!need(1, 2) || (s.params[0] & 3u) || s.params[0] + 4 > eb(0))
            return fail(BGR_ERR_INVALID_ARGUMENT, "u32 system binds {C} with params {aligned byte_offset, k}");
        break;
    case BGR_SYS_U32_STORE_CALL_COUNT:
        if (!need(1, 1) || (s.params[0] & 3u) || s.params[0] + 4 > eb(0))
            return fail(BGR_ERR_INVALID_ARGUMENT, "store_call_count binds {C} with params {aligned byte_offset}");
        break;
    case BGR_SYS_PARTICLES_SPAWN:
        if (!need(3, 4) || eb(0) != 40 || eb(1) != 12 || eb(2) != 8)
            return fail(BGR_ERR_INVALID_ARGUMENT, "spawn_particles binds {Transform(40B), Velocity(12B), Ttl(8B)} with params {rate, ttl, seed_lo, seed_hi}");
        if (e->spawn_sys >= 0) return fail(BGR_ERR_INVALID_ARGUMENT, "spawn_particles registered twice");
        // A shard appends rows locally: the RollbackOrdered index order_base + row of a newborn would collide with the
        // next shard's range, and every shard would draw the same ParticleRng stream.  Dynamic spawning needs one GPU.
        if ((e->cfg.flags & BGR_CFG_SHARDED) || e->cfg.order_base != 0)
            return fail(BGR_ERR_UNSUPPORTED, "spawn_particles is not supported on a sharded engine (BGR_CFG_SHARDED / order_base != 0)");
        if (s.params[0] == 0 || s.params[0] > 4096) return fail(BGR_ERR_INVALID_ARGUMENT, "spawn rate must be in 1..4096");
        e->spawn_sys = int(e->systems.size());
        e->st.rng.seed_from_u64(uint64_t(s.params[2]) | (uint64_t(s.params[3]) << 32));  // insert_resource(ParticleRng(seed_from_u64(seed)))
        break;
    case BGR_SYS_BOX_MOVE:
        if (!need(2, 0) || eb(0) != 40 || eb(1) != 12)
            return fail(BGR_ERR_INVALID_ARGUMENT, "move_cube_system binds {Transform(40B), Velocity(12B)}");
        break;
    case BGR_SYS_DESPAWN_ON_INPUT:
        if (!need(1, 2) || s.params[0] >= BGR_MAX_PLAYERS || s.params[1] > 0xFF)
            return fail(BGR_ERR_INVALID_ARGUMENT, "despawn_on_input binds {C} with params {player_handle < 8, value <= 255}");
        break;
    default: return fail(BGR_ERR_INVALID_ARGUMENT, "unknown system id");
    }
    e->systems.push_back(std::move(s));
    return BGR_OK;
}

BGR_API int bgr_add_user_system(bgr_engine* e, const char* name, const char* cuda_source, const uint32_t* columns,
                                uint32_t n_columns, const uint32_t* params, uint32_t n_params) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    if (e->built) return fail(BGR_ERR_STATE, "systems must be added before bgr_build");
    bool ident = name && *name && !(*name >= '0' && *name <= '9');
    for (const char* q = name; ident && *q; ++q)
        ident = (*q >= 'a' && *q <= 'z') || (*q >= 'A' && *q <= 'Z') || (*q >= '0' && *q <= '9') || *q == '_';
    if (!ident) return fail(BGR_ERR_INVALID_ARGUMENT, "user system name must be a C identifier");
    for (const SystemReg& sy : e->systems)
        if (sy.id == kSysUser && sy.name == name) return fail(BGR_ERR_INVALID_ARGUMENT, std::string("user system '") + name + "' added twice");
    if (!cuda_source) return fail(BGR_ERR_INVALID_ARGUMENT, "null user system source");
    if (std::strlen(cuda_source) > 65536) return fail(BGR_ERR_INVALID_ARGUMENT, "user system source is larger than 64 KB");
    if (n_columns < 1 || n_columns > 4 || !columns) return fail(BGR_ERR_INVALID_ARGUMENT, "a user system binds 1 to 4 columns");
    if (n_params > 8 || (n_params && !params)) return fail(BGR_ERR_INVALID_ARGUMENT, "a user system takes at most 8 parameters");
    SystemReg s;
    s.id = kSysUser;
    for (uint32_t i = 0; i < n_columns; ++i) {
        if (columns[i] >= e->cols.size()) return fail(BGR_ERR_INVALID_ARGUMENT, "system binds an unknown column");
        for (uint32_t c : s.cols)
            if (c == columns[i]) return fail(BGR_ERR_INVALID_ARGUMENT, "a user system binds the same column twice");
        s.cols.push_back(columns[i]);
    }
    s.params.assign(params, params + n_params);
    if (e->systems.size() >= size_t(kMaxGenericSys))
        return fail(BGR_ERR_CAPACITY, "a registration with user systems holds at most 8 systems in total");
    s.name = name;
    s.source = cuda_source;
    e->systems.push_back(std::move(s));
    return BGR_OK;
}

BGR_API int bgr_build(bgr_engine* e) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    if (e->built) return fail(BGR_ERR_STATE, "bgr_build called twice");
    const bool user = has_user_systems(e->systems);
    if (user) {  // user systems run on the registration's own kernel only (generic_program_jit.cuh)
        uint32_t words = 0;
        for (const Column& c : e->cols) words += c.words;
        if (e->systems.size() > size_t(kMaxGenericSys))
            return fail(BGR_ERR_CAPACITY, "a registration with user systems holds at most 8 systems in total");
        if (e->spawn_sys >= 0)
            return fail(BGR_ERR_UNSUPPORTED, "user systems cannot be combined with spawn_particles (spawning runs on the stepwise and bundle paths)");
        if (e->cfg.flags & BGR_CFG_FORCE_STEPWISE)
            return fail(BGR_ERR_UNSUPPORTED, "user systems cannot run with BGR_CFG_FORCE_STEPWISE: they only run on the generated kernel");
        if (e->tune_jit == 0 || e->tune_generic == 0)
            return fail(BGR_ERR_UNSUPPORTED, "user systems need the generated kernel (BGR_TUNE_JIT=0 or BGR_TUNE_GENERIC=0 disables it)");
        if (words > 24)
            return fail(BGR_ERR_UNSUPPORTED, "user systems need a row of at most 24 words (96 bytes of registered columns)");
    }
    CUDA_TRY(cudaSetDevice(e->cfg.device));
    uint32_t plane = 0;
    e->n_ck = 0;
    for (Column& c : e->cols) {
        c.first_plane = plane;
        plane += c.words;
        if (c.hash_kind != BGR_HASH_NONE) {
            if (e->n_ck >= BGR_MAX_CHECKSUM_COLUMNS) return fail(BGR_ERR_CAPACITY, "too many checksummed columns");
            c.ck_slot = int(e->n_ck++);
        }
    }
    e->words = plane;
    e->epad = (e->cfg.max_entities + kTileRows - 1) / kTileRows * kTileRows;
    e->n_tiles_cap = e->epad / kTileRows;
    e->tile_bytes = tile_bytes_of(e->words);
    e->image_bytes = (size_t(e->n_tiles_cap) * e->tile_bytes + 255u) & ~size_t(255);  // ops address images in 256-byte units
    if ((e->image_bytes * (size_t(e->cfg.max_depth) + 1u)) >> 8 > 0xffffffffull)
        return fail(BGR_ERR_CAPACITY, "arena larger than 1 TB");
    size_t total = e->image_bytes * (size_t(e->cfg.max_depth) + 1u);
    CUDA_TRY(cudaMalloc(&e->arena, total));
    CUDA_TRY(cudaMemsetAsync(e->arena, 0, total, e->stream));
    CUDA_TRY(cudaMalloc(&e->d_kill, e->epad));
    CUDA_TRY(cudaMemsetAsync(e->d_kill, 0, e->epad, e->stream));
    const size_t acc_bytes = sizeof(unsigned long long) * kMaxSaves * kAccStride;
    CUDA_TRY(cudaMalloc(&e->d_accum, acc_bytes * bgr_engine::kMaxChains));
    CUDA_TRY(cudaMemsetAsync(e->d_accum, 0, acc_bytes * bgr_engine::kMaxChains, e->stream));
    CUDA_TRY(cudaMalloc(&e->d_ticket, 4 * sizeof(unsigned int) * bgr_engine::kMaxChains));
    CUDA_TRY(cudaMemsetAsync(e->d_ticket, 0, 4 * sizeof(unsigned int) * bgr_engine::kMaxChains, e->stream));
    for (int c = 0; c < bgr_engine::kMaxChains; ++c) {
        e->d_accum_c[c] = e->d_accum + size_t(c) * kMaxSaves * kAccStride;
        e->d_ticket_c[c] = e->d_ticket + 4 * c;
    }
    if (e->tune_tiledep) {
        const size_t nt = size_t(e->tiles_for(e->cfg.max_entities)) + 1;
        CUDA_TRY(cudaMalloc(&e->d_tile_done, nt * sizeof(unsigned int)));
        CUDA_TRY(cudaMalloc(&e->d_tile_cnt, nt * sizeof(unsigned int)));
        CUDA_TRY(cudaMemsetAsync(e->d_tile_done, 0, nt * sizeof(unsigned int), e->stream));
        CUDA_TRY(cudaMemsetAsync(e->d_tile_cnt, 0, nt * sizeof(unsigned int), e->stream));
    }
    if (e->n_chains > 1) {
        for (int c = 0; c < e->n_chains; ++c) {
            CUDA_TRY(cudaStreamCreateWithFlags(&e->chain_stream[c], cudaStreamNonBlocking));
            CUDA_TRY(cudaEventCreateWithFlags(&e->chain_ev[c], cudaEventDisableTiming));
        }
        CUDA_TRY(cudaEventCreateWithFlags(&e->main_ev, cudaEventDisableTiming));
        e->main_dirty = true;  // the memsets above
    }
    for (int i = 0; i < bgr_engine::kBufs; ++i) {
        const size_t out_bytes = sizeof(unsigned long long) * kResultStride * bgr_engine::kMaxChains;
        CUDA_TRY(cudaHostAlloc(&e->h_out[i], out_bytes, cudaHostAllocMapped));
        std::memset(e->h_out[i], 0, out_bytes);
        CUDA_TRY(cudaHostGetDevicePointer(&e->d_out[i], e->h_out[i], 0));
        CUDA_TRY(cudaEventCreateWithFlags(&e->ev[i], cudaEventDisableTiming));
    }
    e->st.ring.reset(e->cfg.max_depth);
    e->st.slot_rows.fill(0);
    e->st.slot_elapsed_ns.fill(0);
    e->st.slot_passive_ver.fill(0);
    if (e->spawn_sys >= 0)
        for (int i = 0; i < bgr_engine::kBufs; ++i) {
            CUDA_TRY(cudaHostAlloc(&e->h_spawn[i], sizeof(float2) * kMaxSpawnVals, cudaHostAllocMapped));
            CUDA_TRY(cudaHostGetDevicePointer(&e->d_spawn[i], e->h_spawn[i], 0));
        }
    detect_bundles(e);
    {   // generic one-launch program: every registered system has a shared-memory implementation, the tile fits twice per SM
        bool ok = e->systems.size() <= size_t(kMaxGenericSys) && e->tile_bytes <= 100u * 1024u;  // at least two blocks per SM
        for (const SystemReg& sy : e->systems)
            ok = ok && (sy.id == BGR_SYS_U32_ADD || sy.id == BGR_SYS_U32_SATSUB_DESPAWN || sy.id == BGR_SYS_U32_STORE_CALL_COUNT ||
                        sy.id == BGR_SYS_PARTICLES_UPDATE || sy.id == BGR_SYS_PARTICLES_DESPAWN || sy.id == BGR_SYS_BOX_MOVE ||
                        sy.id == BGR_SYS_DESPAWN_ON_INPUT || sy.id == kSysUser);
        e->generic_ok = ok;
    }
    const int jrc = jit_specialise(e);
    if (jrc != BGR_OK) return jrc;
    if (user && !e->jit.fn) return fail(BGR_ERR_UNSUPPORTED, "user systems: the generated kernel was not compiled");
    if (e->jit.fn && e->tune_jit_tiledep) {
        const size_t ni = size_t(e->tiles_for(e->cfg.max_entities)) * 4 + 4;
        CUDA_TRY(cudaMalloc(&e->d_item_done, ni * sizeof(unsigned int)));
        CUDA_TRY(cudaMemsetAsync(e->d_item_done, 0, ni * sizeof(unsigned int), e->stream));
    }
    {   // TMA copy kernel: up to six one-tile stages in ~200 KB of shared memory, at least two
        uint32_t st = uint32_t(std::min<size_t>((200u * 1024u) / e->tile_bytes, size_t(kTmaMaxStages)));
        if (env_int("BGR_TUNE_TMA_STAGES", 0) > 0) st = std::min(st, uint32_t(env_int("BGR_TUNE_TMA_STAGES", 0)));
        e->tma_stage_tiles = st >= 2 ? st : 0;
        if (e->tma_stage_tiles) {
            size_t smem = size_t(e->tma_stage_tiles) * e->tile_bytes;
            CUDA_TRY(cudaFuncSetAttribute(k_image_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
            CUDA_TRY(cudaMalloc(&e->d_tma_ticket, 4 * sizeof(unsigned int)));
            CUDA_TRY(cudaMemsetAsync(e->d_tma_ticket, 0, 4 * sizeof(unsigned int), e->stream));
        }
    }
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    e->built = true;
    return BGR_OK;
}

BGR_API int bgr_run_startup_system(bgr_engine* e, uint32_t system) {
    if (!e || !e->built) return fail(BGR_ERR_STATE, "engine not built");
    if (system != BGR_SYS_PARTICLES_SPAWN || e->spawn_sys < 0)
        return fail(BGR_ERR_INVALID_ARGUMENT, "only a registered spawn_particles system can run at Startup");
    int rc = drain(e);
    if (rc != BGR_OK) return rc;
    const SystemReg& sy = e->systems[size_t(e->spawn_sys)];
    const uint32_t rate = sy.params[0];
    if (uint64_t(e->st.n_rows) + rate > e->cfg.max_entities) return fail(BGR_ERR_CAPACITY, "spawn_particles exceeds max_entities");
    for (uint32_t k = 0; k < rate; ++k) {
        e->h_spawn[0][k].x = e->st.rng.random_range(-200.0f, 200.0f);
        e->h_spawn[0][k].y = e->st.rng.random_range(-200.0f, 200.0f);
    }
    const uint64_t ttl = sy.params[1];
    k_sys_particles_spawn<<<e->grid_for(rate, 256), 256, 0, e->stream>>>(
        e->image(0), e->words, e->cols[sy.cols[0]].first_plane, e->cols[sy.cols[1]].first_plane, e->cols[sy.cols[2]].first_plane,
        e->st.n_rows, rate, e->d_spawn[0], uint32_t(ttl), uint32_t(ttl >> 32));
    e->launches += 1;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    e->st.n_rows += rate;
    e->st.live_passive_ver = ++e->st.ver_counter;
    return BGR_OK;
}

BGR_API int bgr_spawn(bgr_engine* e, uint32_t count, uint32_t* first_row_out) {
    if (!e || !e->built) return fail(BGR_ERR_STATE, "engine not built");
    int rc = drain(e);
    if (rc != BGR_OK) return rc;
    if (uint64_t(e->st.n_rows) + count > e->cfg.max_entities) return fail(BGR_ERR_CAPACITY, "spawn exceeds max_entities");
    if (count && e->ticked && ((e->cfg.flags & BGR_CFG_SHARDED) || e->cfg.order_base != 0))
        return fail(BGR_ERR_UNSUPPORTED, "bgr_spawn after the initial population is not supported on a sharded engine "
                                         "(the new rows' RollbackOrdered indices would collide with the next shard's range)");
    uint32_t first = e->st.n_rows;
    if (count) {
        k_spawn_rows<<<e->grid_for(count, 64), 256, 0, e->stream>>>(e->image(0), e->words, first, count);
        e->launches += 1;
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaStreamSynchronize(e->stream));
    }
    e->st.n_rows += count;
    e->st.live_passive_ver = ++e->st.ver_counter;
    if (first_row_out) *first_row_out = first;
    return BGR_OK;
}

BGR_API int bgr_despawn(bgr_engine* e, uint32_t row) {
    if (!e || !e->built) return fail(BGR_ERR_STATE, "engine not built");
    int rc = drain(e);
    if (rc != BGR_OK) return rc;
    if (row >= e->st.n_rows) return fail(BGR_ERR_INVALID_ARGUMENT, "row out of range");
    k_set_alive<<<1, 1, 0, e->stream>>>(e->image(0), e->words, row, 0);
    e->launches += 1;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    return BGR_OK;
}

BGR_API int bgr_row_count(bgr_engine* e, uint32_t* rows_out) {
    if (!e || !rows_out) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    *rows_out = e->st.n_rows;
    return BGR_OK;
}

BGR_API int bgr_active_count(bgr_engine* e, uint64_t* active_out) {
    if (!e || !e->built || !active_out) return fail(BGR_ERR_STATE, "engine not built");
    std::vector<uint8_t> a(e->st.n_rows);
    int rc = read_alive_image(e, 0, 0, e->st.n_rows, e->st.n_rows, a.data());
    if (rc != BGR_OK) return rc;
    uint64_t n = 0;
    for (uint8_t v : a) n += v ? 1 : 0;
    *active_out = n;
    return BGR_OK;
}

BGR_API int bgr_write_component(bgr_engine* e, uint32_t column, uint32_t first_row, uint32_t count, const void* host_src,
                                uint32_t stride) {
    if (!host_src && count) return fail(BGR_ERR_INVALID_ARGUMENT, "null host buffer");
    return transfer_column(e, 0, column, first_row, count, const_cast<void*>(host_src), stride, true);
}

BGR_API int bgr_read_component(bgr_engine* e, uint32_t column, uint32_t first_row, uint32_t count, void* host_dst,
                               uint32_t stride) {
    if (!host_dst && count) return fail(BGR_ERR_INVALID_ARGUMENT, "null host buffer");
    return transfer_column(e, 0, column, first_row, count, host_dst, stride, false);
}

static int presence_args(bgr_engine* e, uint32_t column, uint32_t row) {
    if (!e || !e->built) return fail(BGR_ERR_STATE, "engine not built");
    if (column >= e->cols.size()) return fail(BGR_ERR_INVALID_ARGUMENT, "unknown column");
    if (!e->cols[column].absent) return fail(BGR_ERR_INVALID_ARGUMENT, "column was not registered with BGR_STRATEGY_OPTIONAL");
    if (row >= e->st.n_rows) return fail(BGR_ERR_INVALID_ARGUMENT, "row out of range");
    return drain(e);
}
BGR_API int bgr_remove_component(bgr_engine* e, uint32_t column, uint32_t row) {
    int rc = presence_args(e, column, row);
    if (rc != BGR_OK) return rc;
    k_set_absent<<<1, 1, 0, e->stream>>>(e->image(0), e->words, row, e->cols[column].absent, 1u);
    e->launches += 1;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    e->st.live_passive_ver = ++e->st.ver_counter;
    return BGR_OK;
}
BGR_API int bgr_insert_component(bgr_engine* e, uint32_t column, uint32_t row, const void* value) {
    if (!value) return fail(BGR_ERR_INVALID_ARGUMENT, "null value");
    int rc = presence_args(e, column, row);
    if (rc != BGR_OK) return rc;
    rc = transfer_column(e, 0, column, row, 1, const_cast<void*>(value), e->cols[column].elem_bytes, true);
    if (rc != BGR_OK) return rc;
    k_set_absent<<<1, 1, 0, e->stream>>>(e->image(0), e->words, row, e->cols[column].absent, 0u);
    e->launches += 1;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    return BGR_OK;
}
BGR_API int bgr_has_component(bgr_engine* e, uint32_t column, uint32_t first_row, uint32_t count, uint8_t* host_dst) {
    if (!e || !e->built || !host_dst) return fail(BGR_ERR_STATE, "engine not built");
    if (column >= e->cols.size()) return fail(BGR_ERR_INVALID_ARGUMENT, "unknown column");
    return read_alive_image(e, 0, first_row, count, e->st.n_rows, host_dst, e->cols[column].absent);
}

BGR_API int bgr_host_alloc(size_t bytes, void** out) {
    if (!out) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    *out = nullptr;
    CUDA_TRY(cudaHostAlloc(out, std::max<size_t>(bytes, 1), cudaHostAllocPortable));
    return BGR_OK;
}
BGR_API int bgr_host_free(void* p) {
    if (p) CUDA_TRY(cudaFreeHost(p));
    return BGR_OK;
}
BGR_API int bgr_download_begin(bgr_engine* e, uint32_t column, uint32_t byte_offset, uint32_t byte_len, uint32_t first_row,
                               uint32_t count, void* host_dst, uint32_t* ticket_out) {
    return download_begin(e, column, byte_offset, byte_len, first_row, count, host_dst, ticket_out);
}
BGR_API int bgr_download_wait(bgr_engine* e, uint32_t ticket) { return download_wait(e, ticket); }

BGR_API int bgr_read_alive(bgr_engine* e, uint32_t first_row, uint32_t count, uint8_t* host_dst) {
    if (!e || !e->built) return fail(BGR_ERR_STATE, "engine not built");
    return read_alive_image(e, 0, first_row, count, e->st.n_rows, host_dst);
}

BGR_API int bgr_rollback_frame_count(bgr_engine* e, int32_t* out) {
    if (!e || !out) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    *out = e->st.frame_count; return BGR_OK;
}
BGR_API int bgr_set_rollback_frame_count(bgr_engine* e, int32_t frame) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    e->st.frame_count = frame; return BGR_OK;
}
BGR_API int bgr_confirmed_frame_count(bgr_engine* e, int32_t* out) {
    if (!e || !out) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    *out = e->st.confirmed; return BGR_OK;
}
BGR_API int bgr_max_prediction_window(bgr_engine* e, uint32_t* out) {
    if (!e || !out) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    *out = e->st.has_maxpred ? e->st.maxpred : 0; return BGR_OK;
}

BGR_API int bgr_set_depth(bgr_engine* e, uint32_t depth) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    e->st.has_maxpred = true; e->st.maxpred = depth;  // MaxPredictionWindow: sync_depth applies it before every save
    e->st.ring.set_depth(depth);
    return BGR_OK;
}
BGR_API int bgr_confirm(bgr_engine* e, int32_t confirmed_frame) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    e->st.confirmed = confirmed_frame;
    e->st.ring.confirm(confirmed_frame);
    return BGR_OK;
}
BGR_API int bgr_snapshot_frames(bgr_engine* e, int32_t* frames_out, uint32_t cap, uint32_t* n_out) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    std::vector<int32_t> f;
    e->st.ring.frames(&f);
    for (uint32_t i = 0; i < f.size() && i < cap && frames_out; ++i) frames_out[i] = f[i];
    if (n_out) *n_out = uint32_t(f.size());
    return BGR_OK;
}

BGR_API int bgr_peek(bgr_engine* e, int32_t frame, uint32_t column, uint32_t first_row, uint32_t count, void* host_dst,
                     uint32_t stride, uint8_t* alive_dst, int32_t* found) {
    if (!e || !e->built || !found) return fail(BGR_ERR_STATE, "engine not built");
    uint32_t slot = 0;
    if (!e->st.ring.peek(frame, &slot)) { *found = 0; return BGR_OK; }
    *found = 1;
    int rc = transfer_column(e, slot + 1, column, first_row, count, host_dst, stride, false);
    if (rc != BGR_OK) return rc;
    // alive_dst[i] = the snapshot of `frame` holds this column for row first_row+i (the row existed and had the component)
    if (alive_dst) return read_alive_image(e, slot + 1, first_row, count, e->st.slot_rows[slot], alive_dst, e->cols[column].absent);
    return BGR_OK;
}

BGR_API int bgr_submit_requests(bgr_engine* e, const bgr_session_info* session, const bgr_request* requests,
                                uint32_t n_requests) {
    return submit(e, session, requests, n_requests);
}

BGR_API int bgr_collect(bgr_engine* e, bgr_checksum* checksums_out, uint32_t checksums_cap, uint32_t* n_checksums_out) {
    return collect(e, checksums_out, checksums_cap, n_checksums_out);
}

BGR_API int bgr_handle_requests(bgr_engine* e, const bgr_session_info* session, const bgr_request* requests,
                                uint32_t n_requests, bgr_checksum* checksums_out, uint32_t checksums_cap,
                                uint32_t* n_checksums_out) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    // the checksums returned must be THIS vector's: earlier bgr_submit_requests have to be collected first
    if (!e->pending.empty())
        return fail(BGR_ERR_STATE, "bgr_handle_requests with un-collected bgr_submit_requests pending: call bgr_collect first");
    e->tiledep_chain = false;
    int rc = submit(e, session, requests, n_requests);
    if (rc != BGR_OK) return rc;
    return collect(e, checksums_out, checksums_cap, n_checksums_out);
}

BGR_API int bgr_save_world(bgr_engine* e, bgr_checksum* checksum_out) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    bgr_request rq;
    std::memset(&rq, 0, sizeof rq);
    rq.kind = BGR_REQ_SAVE; rq.frame = e->st.frame_count;
    uint32_t n = 0;
    return bgr_handle_requests(e, nullptr, &rq, 1, checksum_out, checksum_out ? 1 : 0, &n);
}

BGR_API int bgr_load_world(bgr_engine* e) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    bgr_request rq;
    std::memset(&rq, 0, sizeof rq);
    rq.kind = BGR_REQ_LOAD; rq.frame = e->st.frame_count;
    uint32_t n = 0;
    return bgr_handle_requests(e, nullptr, &rq, 1, nullptr, 0, &n);
}

BGR_API int bgr_advance_world(bgr_engine* e, const uint8_t* inputs, const uint8_t* status, uint32_t n_players) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    if (n_players > BGR_MAX_PLAYERS) return fail(BGR_ERR_INVALID_ARGUMENT, "n_players > BGR_MAX_PLAYERS");
    bgr_request rq;
    std::memset(&rq, 0, sizeof rq);
    rq.kind = kReqAdvanceNoBump; rq.n_players = n_players;
    for (uint32_t i = 0; i < n_players; ++i) { rq.inputs[i] = inputs ? inputs[i] : 0; rq.status[i] = status ? status[i] : 0; }
    uint32_t n = 0;
    return bgr_handle_requests(e, nullptr, &rq, 1, nullptr, 0, &n);
}

BGR_API int bgr_last_partials(bgr_engine* e, bgr_partial* out, uint32_t cap, uint32_t* n_out) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    for (uint32_t i = 0; i < e->last_partials.size() && i < cap && out; ++i) out[i] = e->last_partials[i];
    if (n_out) *n_out = uint32_t(e->last_partials.size());
    return BGR_OK;
}

BGR_API int bgr_fold_partials(const bgr_partial* combined, bgr_checksum* out) {
    if (!combined || !out) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    fold(*combined, out);
    return BGR_OK;
}

BGR_API int bgr_collect_partials(bgr_engine* e, bgr_partial* partials_out, uint32_t cap, uint32_t* n_out) {
    uint32_t n = 0;
    int rc = collect(e, nullptr, 0, &n);
    if (rc != BGR_OK) return rc;
    for (uint32_t i = 0; i < n && i < cap && partials_out; ++i) partials_out[i] = e->last_partials[i];
    if (n_out) *n_out = n;
    return BGR_OK;
}

BGR_API int bgr_fold_partials_n(const bgr_partial* combined, uint32_t n, bgr_checksum* out) {
    if ((!combined || !out) && n) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    for (uint32_t i = 0; i < n; ++i) fold(combined[i], &out[i]);
    return BGR_OK;
}

BGR_API uint64_t bgr_seahash(const void* bytes, uint64_t len) {
    const uint8_t* p = static_cast<const uint8_t*>(bytes);
    uint64_t a = kSeaA, b = kSeaB, c = kSeaC, d = kSeaD;
    uint64_t i = 0;
    for (; i + 8 <= len; i += 8) {
        uint64_t w;
        std::memcpy(&w, p + i, 8);  // little-endian host
        uint64_t t = sea_diffuse(a ^ w);
        a = b; b = c; c = d; d = t;
    }
    if (i < len) {
        uint64_t w = 0;
        std::memcpy(&w, p + i, size_t(len - i));
        a = sea_diffuse(a ^ w);
    }
    return sea_diffuse(a ^ b ^ c ^ d ^ len);
}

// the engine's ParticleRng arithmetic on its own (host only): known-answer tests of SplitMix64 / xoshiro256++ / the
// f32 range sampling run against exactly the code that spawn_particles uses
BGR_API int bgr_particle_rng_stream(uint64_t seed, const uint64_t* state4_or_null, uint32_t n, uint64_t* next_u64_out,
                                    float* range_out, float low, float high) {
    ParticleRng a, b;
    if (state4_or_null) { for (int i = 0; i < 4; ++i) a.s[i] = b.s[i] = state4_or_null[i]; }
    else { a.seed_from_u64(seed); b.seed_from_u64(seed); }
    for (uint32_t i = 0; i < n; ++i) {
        if (next_u64_out) next_u64_out[i] = a.next_u64();
        if (range_out) range_out[i] = b.random_range(low, high);
    }
    return BGR_OK;
}
BGR_API int bgr_splitmix64_stream(uint64_t seed, uint32_t n, uint64_t* out) {
    if (!out && n) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    SplitMix64 sm{seed};
    for (uint32_t i = 0; i < n; ++i) out[i] = sm.next_u64();
    return BGR_OK;
}

BGR_API uint32_t bgr_ggrs_time_delta_bits(uint32_t fps, int32_t frame) {
    if (fps == 0) return 0;
    uint64_t f = uint64_t(int64_t(frame));
    uint64_t now = f * 1000000000ULL / fps, prev = (f - 1) * 1000000000ULL / fps;
    return f32_bits(duration_as_secs_f32(now - prev));
}

BGR_API int bgr_launch_count(bgr_engine* e, uint64_t* out) {
    if (!e || !out) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    *out = e->launches; return BGR_OK;
}
BGR_API int bgr_slot_bytes(bgr_engine* e, uint64_t* out) {
    if (!e || !out) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    *out = uint64_t(e->st.n_rows) * (uint64_t(e->words) * 4u + 1u); return BGR_OK;
}
BGR_API int bgr_generic_specialised(bgr_engine* e, uint32_t* specialised_out) {
    if (!e || !specialised_out) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    *specialised_out = e->jit.fn ? 1u : 0u;
    return BGR_OK;
}
BGR_API int bgr_last_path(bgr_engine* e, uint32_t* fused_out) {
    if (!e || !fused_out) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    *fused_out = e->last_fused ? 1u : 0u; return BGR_OK;
}
BGR_API int bgr_synchronize(bgr_engine* e) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    return BGR_OK;
}


// ---- shard group (multi-GPU cross-shard exchange inside the engine; shard_group.hpp) ----
BGR_API int bgr_shard_group_join(bgr_engine* e, const char* name, uint32_t rank, uint32_t world_size, uint32_t timeout_ms) {
    if (!e || !e->built) return fail(BGR_ERR_STATE, "engine not built");
    if (!name || !*name) return fail(BGR_ERR_INVALID_ARGUMENT, "null group name");
    if (!(e->cfg.flags & BGR_CFG_SHARDED)) return fail(BGR_ERR_STATE, "only a BGR_CFG_SHARDED engine can join a shard group");
    if (e->group) return fail(BGR_ERR_STATE, "engine is already in a shard group");
    if (!e->pending.empty()) return fail(BGR_ERR_STATE, "collect every submitted request vector before joining a shard group");
    if (e->n_chains != 1) return fail(BGR_ERR_UNSUPPORTED, "BGR_TUNE_CHAINS > 1 cannot be combined with a shard group");
    CUDA_TRY(cudaSetDevice(e->cfg.device));
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    auto* g = new ShardGroup();
    if (timeout_ms) g->timeout_ms = timeout_ms;
    std::string err;
    const uint32_t block_words = uint32_t(kResultStride) * bgr_engine::kMaxChains;
    static_assert(bgr_engine::kBufs == int(kGroupBufs) && kMaxSaves == int(kGroupMaxSaves) && kAccStride == int(kGroupAccStride),
                  "shard_group.hpp mirrors the engine's result block layout");
    if (!g->join(name, rank, world_size, block_words, e->seq, &err)) { delete g; return fail(BGR_ERR_STATE, err); }
    // the block area becomes page-locked and visible to this GPU: the fused kernel's last block stores its result rows there
    cudaError_t ce = cudaHostRegister(g->blocks_base(), g->blocks_bytes(), cudaHostRegisterMapped | cudaHostRegisterPortable);
    if (ce != cudaSuccess) { delete g; return fail(BGR_ERR_CUDA, std::string("cudaHostRegister(shard group segment): ") + cudaGetErrorString(ce)); }
    for (int b = 0; b < bgr_engine::kBufs; ++b) {
        e->own_h_out[b] = e->h_out[b]; e->own_d_out[b] = e->d_out[b];
        e->h_out[b] = reinterpret_cast<unsigned long long*>(g->block(rank, uint32_t(b)));
        void* dp = nullptr;
        ce = cudaHostGetDevicePointer(&dp, e->h_out[b], 0);
        if (ce != cudaSuccess) {
            for (int k = 0; k <= b; ++k) { e->h_out[k] = e->own_h_out[k]; e->d_out[k] = e->own_d_out[k]; }
            cudaHostUnregister(g->blocks_base());
            delete g;
            return fail(BGR_ERR_CUDA, std::string("cudaHostGetDevicePointer: ") + cudaGetErrorString(ce));
        }
        e->d_out[b] = static_cast<unsigned long long*>(dp);
    }
    e->group = g;
    e->gseq = 0;
    e->next_buf = 0;
    return BGR_OK;
}

BGR_API int bgr_shard_group_leave(bgr_engine* e) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    if (!e->group) return BGR_OK;
    if (!e->pending.empty()) return fail(BGR_ERR_STATE, "collect every submitted request vector before leaving the shard group");
    cudaSetDevice(e->cfg.device);
    cudaStreamSynchronize(e->stream);
    cudaHostUnregister(e->group->blocks_base());
    for (int b = 0; b < bgr_engine::kBufs; ++b) { e->h_out[b] = e->own_h_out[b]; e->d_out[b] = e->own_d_out[b]; }
    delete e->group;
    e->group = nullptr;
    return BGR_OK;
}

// the group's host logic on its own (no GPU): CPU tests drive join / publish / collect with a stand-in for the kernel's publish
struct bgr_group { ShardGroup g; uint32_t n_columns = 0; };
BGR_API bgr_group* bgr_group_join(const char* name, uint32_t rank, uint32_t world_size, uint32_t n_columns, uint32_t timeout_ms) {
    if (!name) { fail(BGR_ERR_INVALID_ARGUMENT, "null group name"); return nullptr; }
    auto* h = new bgr_group();
    h->n_columns = n_columns;
    if (timeout_ms) h->g.timeout_ms = timeout_ms;
    std::string err;
    if (!h->g.join(name, rank, world_size, uint32_t(kResultStride) * bgr_engine::kMaxChains, 0, &err)) { fail(BGR_ERR_STATE, err); delete h; return nullptr; }
    return h;
}
BGR_API void bgr_group_leave(bgr_group* h) { delete h; }
BGR_API int bgr_group_publish(bgr_group* h, uint64_t gseq, const bgr_partial* partials, uint32_t n) {
    if (!h || (!partials && n) || gseq == 0 || n > uint32_t(kMaxSaves)) return fail(BGR_ERR_INVALID_ARGUMENT, "bad argument");
    std::string err;
    if (!h->g.wait_reusable(gseq, &err)) return fail(BGR_ERR_STATE, err);
    int32_t frames[kMaxSaves]; uint32_t totals[kMaxSaves];
    for (uint32_t k = 0; k < n; ++k) { frames[k] = partials[k].frame; totals[k] = uint32_t(partials[k].total); }
    h->g.publish_meta(gseq, n, h->n_columns, frames, totals);
    h->g.publish_block_from_host(gseq, partials, n);
    return BGR_OK;
}
BGR_API int bgr_group_collect(bgr_group* h, uint64_t gseq, bgr_checksum* out, uint32_t cap, uint32_t* n_out) {
    if (!h || gseq == 0) return fail(BGR_ERR_INVALID_ARGUMENT, "bad argument");
    bgr_partial combined[kMaxSaves];
    uint32_t n = 0;
    uint64_t flags = 0;
    std::string err;
    if (!h->g.combine(gseq, combined, kMaxSaves, &n, &flags, &err)) return fail(BGR_ERR_STATE, err);
    for (uint32_t k = 0; k < n && k < cap && out; ++k) fold(combined[k], &out[k]);
    if (n_out) *n_out = n;
    return BGR_OK;
}

// No session (schedule_systems.rs:70-79): "reset time data and snapshots" — the frame resources go back to their
// session-less values; the caller (run_ggrs_schedules' mirror) also clears LocalPlayers and its accumulator.
BGR_API int bgr_reset_session(bgr_engine* e) {
    if (!e) return fail(BGR_ERR_INVALID_ARGUMENT, "null engine");
    if (!e->pending.empty()) return fail(BGR_ERR_STATE, "collect every submitted request vector first");
    e->st.frame_count = 0;        // RollbackFrameCount(0)
    e->st.confirmed = -1;         // ConfirmedFrameCount(-1)
    e->st.has_maxpred = true;     // MaxPredictionWindow(8)
    e->st.maxpred = 8;
    return BGR_OK;
}

BGR_API int bgr_host_profile(bgr_engine* e, uint64_t* out, uint32_t cap) {
    if (!e || !out) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    for (uint32_t i = 0; i < cap && i < 8; ++i) out[i] = e->prof[i];
    return BGR_OK;
}

BGR_API int bgr_stream(bgr_engine* e, void** stream_out) {
    if (!e || !stream_out) return fail(BGR_ERR_INVALID_ARGUMENT, "null argument");
    *stream_out = e->stream;
    return BGR_OK;
}

// Device-side launch trace: every fused launch records when its first block started and when its last block
// finished (ns of the GPU's globaltimer) — the evidence for overlapping consecutive ticks (DESIGN.md) when no
// system profiler is available.  Two atomics per block; off unless enabled.
BGR_API int bgr_trace_enable(bgr_engine* e, uint32_t capacity) {
    if (!e || !e->built) return fail(BGR_ERR_STATE, "engine not built");
    int rc = drain(e);
    if (rc != BGR_OK) return rc;
    if (e->d_trace) { CUDA_TRY(cudaFree(e->d_trace)); e->d_trace = nullptr; e->trace_cap = 0; }
    if (capacity == 0) return BGR_OK;
    std::vector<unsigned long long> init(size_t(capacity) * 4, 0ULL);
    for (uint32_t i = 0; i < capacity; ++i) init[4 * i] = ~0ULL;
    CUDA_TRY(cudaMalloc(&e->d_trace, init.size() * sizeof(unsigned long long)));
    CUDA_TRY(cudaMemcpy(e->d_trace, init.data(), init.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice));
    e->trace_cap = capacity;
    e->trace_first_seq = e->seq + 1;
    return BGR_OK;
}
BGR_API int bgr_trace_read(bgr_engine* e, uint64_t* start_end_ns_out, uint32_t cap, uint32_t* n_out) {
    if (!e || !e->d_trace) return fail(BGR_ERR_STATE, "trace not enabled");
    int rc = drain(e);
    if (rc != BGR_OK) return rc;
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    const uint64_t done = e->seq + 1 > e->trace_first_seq ? e->seq + 1 - e->trace_first_seq : 0;
    const uint32_t n = uint32_t(std::min<uint64_t>(std::min<uint64_t>(done, e->trace_cap), cap));
    if (n && start_end_ns_out) CUDA_TRY(cudaMemcpy(start_end_ns_out, e->d_trace, size_t(n) * 4 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    if (n_out) *n_out = n;
    return BGR_OK;
}

// ---- host-side ring bookkeeping on its own (pure host logic; used by the "not gpu" KAT tests) ----
struct bgr_ring { SlotRing r; };
BGR_API bgr_ring* bgr_ring_create(uint32_t n_slots) { auto* r = new bgr_ring(); r->r.reset(n_slots); return r; }
BGR_API void bgr_ring_destroy(bgr_ring* r) { delete r; }
BGR_API uint32_t bgr_ring_depth(bgr_ring* r) { return r->r.depth(); }
BGR_API int bgr_ring_set_depth(bgr_ring* r, uint32_t depth) { r->r.set_depth(depth); return BGR_OK; }
BGR_API int bgr_ring_push(bgr_ring* r, int32_t frame, uint32_t* slot_out) {
    uint32_t s = r->r.push(frame);
    if (s == SlotRing::kNoSlot) return fail(BGR_ERR_CAPACITY, "ring out of slots");
    if (slot_out) *slot_out = s;
    return BGR_OK;
}
BGR_API int bgr_ring_confirm(bgr_ring* r, int32_t frame) { r->r.confirm(frame); return BGR_OK; }
BGR_API int bgr_ring_rollback(bgr_ring* r, int32_t frame, uint32_t* slot_out) {
    std::string err;
    if (!r->r.rollback(frame, &err)) return fail(BGR_ERR_NO_SNAPSHOT, err);
    uint32_t s = 0;
    r->r.get(&s, nullptr);
    if (slot_out) *slot_out = s;
    return BGR_OK;
}
BGR_API int bgr_ring_get(bgr_ring* r, uint32_t* slot_out) {
    std::string err;
    uint32_t s = 0;
    if (!r->r.get(&s, &err)) return fail(BGR_ERR_NO_SNAPSHOT, err);
    if (slot_out) *slot_out = s;
    return BGR_OK;
}
BGR_API int bgr_ring_peek(bgr_ring* r, int32_t frame, uint32_t* slot_out, int32_t* found) {
    uint32_t s = 0;
    bool ok = r->r.peek(frame, &s);
    if (found) *found = ok ? 1 : 0;
    if (ok && slot_out) *slot_out = s;
    return BGR_OK;
}

}  // extern "C"
