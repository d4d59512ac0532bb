// k_generic_program SPECIALISED AT RUN TIME for one registration (compiled by NVRTC inside bgr_build: engine.cu `jit_specialise`, jit.hpp).
//
// The interpreter (generic_program.cuh) reads the schema — which planes a system touches, which byte ranges are hashed —
// from its parameter block, so a tile has to live in shared memory (registers cannot be indexed at run time; the
// register-resident attempts with select chains / jump tables are recorded in DESIGN.md).  With the schema as
// COMPILE-TIME constants every plane index is a literal, and the same program becomes what k_particles_program is for
// the particles bundle:
//
//     LOAD / first read : coalesced ld.global of the row's words, plane by plane, from the slot / live image
//     ADVANCE           : the registered systems update the register copy (indices are constants: plain register ops)
//     SAVE              : coalesced st.global of the words to the frame's slot + the per-entity seahash of every
//                         checksummed column, folded warp-REDUX -> shared atomics like the interpreter
//     end               : st.global to the live image
//
// no shared-memory tile, no bulk copy, no block barrier inside a tile's program, no spec decoding.  The engine generates
// a prelude of #defines (BGR_JIT_*) from the registration and compiles prelude + this file; parameter block, result
// protocol, tile claiming and op semantics are the interpreter's, and every parity test of the generic path runs on
// both (BGR_TUNE_JIT=0 / 2).
//
// Reference semantics: handle_requests (schedule_systems.rs:170-289) over ComponentSnapshotPlugin::save / load
// (component_snapshot.rs:66-123) and the checksum plugins (component_checksum.rs:67-108).
#pragma once
#include "generic_program.cuh"

namespace bgr {

constexpr int kJitWords = BGR_JIT_WORDS;  // word planes per row
constexpr int kJitRows = BGR_JIT_ROWS;    // rows of a work item per thread
// rows per WORK ITEM: a tile (512) for worlds of many tiles per SM; 256 / 128 for small worlds — 100k entities are 196 tiles on
// 148 SMs, so with whole tiles a third of the SMs carry two tiles and set the kernel's duration (they are bound by the integer
// multiply pipe of the seahash, scripts/frame_cost_fit.py) while the others idle half of it; quarter tiles spread the rows evenly
constexpr int kJitItemRows = BGR_JIT_ITEM_ROWS;
constexpr int kJitSubs = int(kTileRows) / kJitItemRows;  // work items per tile
constexpr int kJitNSys = BGR_JIT_NSYS;
constexpr int kJitNHash = BGR_JIT_NHASH;
constexpr SysSpec kJitSys[kJitNSys + 1] = {BGR_JIT_SYS_LIST};      // {id, plane0, plane1, need, param}, ... + one dummy
constexpr HashSpec kJitHash[kJitNHash + 1] = {BGR_JIT_HASH_LIST};  // {first_plane, off, len, finite, slot, absent}, ... + one dummy

// seahash of the NWORDS whole words at planes [F, F + NWORDS) of a row: the stream form of seahash.cuh with the lane
// rotation done by renaming (word pair q goes to lane q % 4, the odd tail word to the next lane)
template <int F, int NWORDS>
__device__ __forceinline__ uint64_t jit_hash_words(const uint32_t (&w)[kJitWords]) {
    uint64_t s[4] = {kSeaA, kSeaB, kSeaC, kSeaD};
#pragma unroll
    for (int q = 0; q < NWORDS / 2; ++q)
        s[q & 3] = sea_diffuse(s[q & 3] ^ (uint64_t(w[F + 2 * q]) | (uint64_t(w[F + 2 * q + 1]) << 32)));
    if (NWORDS & 1) s[(NWORDS / 2) & 3] = sea_diffuse(s[(NWORDS / 2) & 3] ^ uint64_t(w[F + NWORDS - 1]));
    return sea_diffuse(s[0] ^ s[1] ^ s[2] ^ s[3] ^ uint64_t(NWORDS * 4));
}

struct JitRows {
    uint32_t w[kJitRows][kJitWords];  // the rows' words
    uint32_t m[kJitRows];             // mask bytes: bit 0 alive, bits 1.. absent bits of the optional columns
    uint64_t t0[kJitRows];            // first lane of the per-entity hash (RollbackOrdered index): once per tile
    bool kill[kJitRows];
};

// the S-th registered system on the register copy; every system sees the entity's presence as it was before the frame
template <int S>
__device__ __forceinline__ void jit_run_systems(JitRows& r, const Op& op, float dt, int32_t frame, unsigned long long row0, int B) {
    if constexpr (S < kJitNSys) {
        constexpr SysSpec sy = kJitSys[S];
#pragma unroll
        for (int k = 0; k < kJitRows; ++k) {
            const bool on = row_matches(r.m[k], sy.need);
            if constexpr (sy.id == BGR_SYS_U32_ADD) {
                r.w[k][sy.plane0] += on ? sy.param : 0u;
            } else if constexpr (sy.id == BGR_SYS_U32_SATSUB_DESPAWN) {
                uint32_t v = r.w[k][sy.plane0];
                v = v > sy.param ? v - sy.param : 0u;
                r.w[k][sy.plane0] = on ? v : r.w[k][sy.plane0];
                r.kill[k] = r.kill[k] || (on && v == 0u);
            } else if constexpr (sy.id == BGR_SYS_U32_STORE_CALL_COUNT) {
                r.w[k][sy.plane0] = on ? op.call_count + sy.param : r.w[k][sy.plane0];
            } else if constexpr (sy.id == BGR_SYS_DESPAWN_ON_INPUT) {  // param = player handle | value << 8
                const uint32_t player = sy.param & 0xFFu, n_players = (op.flags >> 8) & 0xFu;
                const uint32_t input = player < n_players && player < 8 ? op.inputs[player] : 0u;
                r.kill[k] = r.kill[k] || (on && input == (sy.param >> 8));
            } else if constexpr (sy.id == BGR_SYS_PARTICLES_UPDATE) {
                uint32_t tx = r.w[k][sy.plane0], ty = r.w[k][sy.plane0 + 1], tz = r.w[k][sy.plane0 + 2];
                uint32_t vx = r.w[k][sy.plane1], vy = r.w[k][sy.plane1 + 1], vz = r.w[k][sy.plane1 + 2];
                particle_step(tx, ty, tz, vx, vy, vz, dt);
                if (on) {
                    r.w[k][sy.plane0] = tx; r.w[k][sy.plane0 + 1] = ty; r.w[k][sy.plane0 + 2] = tz;
                    r.w[k][sy.plane1] = vx; r.w[k][sy.plane1 + 1] = vy; r.w[k][sy.plane1 + 2] = vz;
                }
            } else if constexpr (sy.id == BGR_SYS_PARTICLES_DESPAWN) {
                uint64_t ttl = (uint64_t(r.w[k][sy.plane0 + 1]) << 32) | r.w[k][sy.plane0];
                ttl -= 1;
                if (on) { r.w[k][sy.plane0] = uint32_t(ttl); r.w[k][sy.plane0 + 1] = uint32_t(ttl >> 32); }
                r.kill[k] = r.kill[k] || (on && ttl == 0);
            } else if constexpr (sy.id == BGR_SYS_BOX_MOVE) {
                if (on) {  // two to four entities: a branch costs nothing and keeps powf off the other rows
                    float tx = __uint_as_float(r.w[k][sy.plane0]), ty = __uint_as_float(r.w[k][sy.plane0 + 1]), tz = __uint_as_float(r.w[k][sy.plane0 + 2]);
                    float vx = __uint_as_float(r.w[k][sy.plane1]), vy = __uint_as_float(r.w[k][sy.plane1 + 1]), vz = __uint_as_float(r.w[k][sy.plane1 + 2]);
                    const unsigned long long handle = row0 + uint32_t(k * B);
                    const uint32_t n_players = (op.flags >> 8) & 0xFu;
                    const uint32_t input = handle < n_players && handle < 8 ? op.inputs[handle] : 0u;
                    box_move_step(tx, ty, tz, vx, vy, vz, dt, input);
                    r.w[k][sy.plane0] = __float_as_uint(tx); r.w[k][sy.plane0 + 1] = __float_as_uint(ty); r.w[k][sy.plane0 + 2] = __float_as_uint(tz);
                    r.w[k][sy.plane1] = __float_as_uint(vx); r.w[k][sy.plane1 + 1] = __float_as_uint(vy); r.w[k][sy.plane1 + 2] = __float_as_uint(vz);
                }
            }
#ifdef BGR_SYS_USER  // the prelude registers user systems (user_system.cuh): param = the system's index among them
            else if constexpr (sy.id == BGR_SYS_USER) {
                bgr_sys_ctx ctx;
                ctx.dt = dt;
                ctx.frame = frame;
                ctx.n_players = (op.flags >> 8) & 0xFu;
#pragma unroll
                for (int j = 0; j < 8; ++j) ctx.inputs[j] = op.inputs[j];
                ctx.order = row0 + uint32_t(k * B);
                ::bgr_user_system<int(sy.param)>::run(r.w[k], on, ctx, r.kill[k]);
            }
#endif
        }
        jit_run_systems<S + 1>(r, op, dt, frame, row0, B);
    }
}

// the C-th checksummed column: per-entity hash of the thread's rows, folded into the save's shared accumulators
template <int C>
__device__ __forceinline__ void jit_hash_columns(const JitRows& r, unsigned int* a, uint32_t lane, uint32_t& bad) {
    if constexpr (C < kJitNHash) {
        constexpr HashSpec hs = kJitHash[C];
        constexpr int F = int(hs.first_plane + (hs.off >> 2)), NWORDS = int(hs.len >> 2);
        uint64_t hx = 0;
#pragma unroll
        for (int k = 0; k < kJitRows; ++k) {
            const bool has = row_matches(r.m[k], hs.absent);  // Query<(&RollbackId, &T)>: exists and has the component
            if constexpr (hs.finite != 0) {
                uint32_t nonfinite = 0;
#pragma unroll
                for (int j = 0; j < NWORDS; ++j) nonfinite |= f32_bits_nonfinite(r.w[k][F + j]);
                bad |= has ? nonfinite : 0u;
            }
            const uint64_t e = sea_hash_entity(r.t0[k], jit_hash_words<F, NWORDS>(r.w[k]));
            hx ^= has ? e : 0ULL;
        }
        const unsigned full = 0xffffffffu;
        const uint32_t lo = __reduce_xor_sync(full, uint32_t(hx)), hi = __reduce_xor_sync(full, uint32_t(hx >> 32));
        if (lane == 0) { atomicXor(&a[2 * hs.slot], lo); atomicXor(&a[2 * hs.slot + 1], hi); }
        jit_hash_columns<C + 1>(r, a, lane, bad);
    }
}

extern "C" __global__ void __launch_bounds__(BGR_JIT_ITEM_ROWS / BGR_JIT_ROWS, BGR_JIT_MINB) k_generic_jit(const __grid_constant__ GenericParams p) {
    constexpr int B = kJitItemRows / kJitRows;  // threads per work item
    __shared__ unsigned int s_acc[kMaxSaves * kAccStride * 2];
    __shared__ uint32_t s_next;
    __shared__ unsigned int s_last;

    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    // Overlap of consecutive request vectors (bgr_submit_requests with others un-collected): work item i of tick k+1 only
    // depends on work item i of tick k.  A signalling launch lets the next one be scheduled as its own blocks retire
    // (griddepcontrol.launch_dependents); a waiting launch was started with programmatic stream serialisation, skips the
    // grid-level wait and instead waits per item for item_done[i] >= wait_seq.  Both grids are at most one wave of resident
    // blocks and every block of the earlier grid has started before the first block of the later one does, so the spin
    // cannot starve what it waits for.  (k_particles_program's protocol, DESIGN.md "Overlapping consecutive ticks".)
    const bool signal_items = (p.flags & PF_TILE_SIGNAL) != 0u, wait_items = (p.flags & PF_TILE_WAIT) != 0u;
    if (signal_items || wait_items) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (p.trace && tid == 0) atomicMin(&p.trace[0], globaltimer_ns());
    for (uint32_t i = tid; i < p.n_saves * kAccStride * 2; i += B) s_acc[i] = 0u;
    if (!wait_items) asm volatile("griddepcontrol.wait;" ::: "memory");  // a no-op unless launched as a programmatic dependent
    __syncthreads();

    const uint8_t* first_img = p.arena + ((p.flags & PF_READ_LIVE) ? size_t(0) : (size_t(p.ops[0].image_off256) << 8));
    const uint32_t first_rows = (p.flags & PF_READ_LIVE) ? p.live_rows : p.ops[0].n_rows;
    constexpr uint32_t kTileBytes = kTileRows * (4u * kJitWords + 1u);
    constexpr uint32_t kAliveOff = uint32_t(kJitWords) * kPlaneBytes;  // the mask bytes follow the word planes inside a tile

    const uint32_t n_items = p.n_tiles * uint32_t(kJitSubs);
    for (uint32_t item = blockIdx.x; item < n_items;) {
        __syncthreads();  // every thread has read the previous s_next
        if (tid == 0) {
            s_next = gridDim.x + atomicAdd(&p.ticket[1], 1u);
            if (wait_items && item < p.wait_items)
                while (int32_t(ld_acquire_gpu(&p.item_done[item]) - p.wait_seq) < 0) {}  // the previous tick's stores of this item are visible
        }
        __syncthreads();
        const uint32_t next_item = s_next;
        const uint32_t tile = item / uint32_t(kJitSubs), sub_row0 = (item % uint32_t(kJitSubs)) * uint32_t(kJitItemRows) + tid;  // first row of the thread inside the tile
        const size_t tile_off = size_t(tile) * kTileBytes;
        const unsigned long long row0 = p.order_base + size_t(tile) * kTileRows + sub_row0;

        JitRows r;
        auto load = [&](const uint8_t* img, uint32_t n_rows_src) {
            const uint8_t* t = img + tile_off;
#pragma unroll
            for (int k = 0; k < kJitRows; ++k) {
                const uint32_t row = sub_row0 + k * B;
#pragma unroll
                for (int j = 0; j < kJitWords; ++j) r.w[k][j] = __ldcg(reinterpret_cast<const uint32_t*>(t + size_t(j) * kPlaneBytes + size_t(row) * 4u));
                const uint32_t mm = __ldcg(t + kAliveOff + row);  // .cg: L2 only — overlapping grids share an SM's L1 without a kernel boundary in between
                r.m[k] = (tile * kTileRows + row < n_rows_src) ? mm : 0u;  // rows the image never contained come back dead
            }
        };
        auto store = [&](uint8_t* img) {
            uint8_t* t = img + tile_off;
#pragma unroll
            for (int k = 0; k < kJitRows; ++k) {
                const uint32_t row = sub_row0 + k * B;
#pragma unroll
                for (int j = 0; j < kJitWords; ++j) *reinterpret_cast<uint32_t*>(t + size_t(j) * kPlaneBytes + size_t(row) * 4u) = r.w[k][j];
                t[kAliveOff + row] = uint8_t(r.m[k]);
            }
        };
        load(first_img, first_rows);
#pragma unroll
        for (int k = 0; k < kJitRows; ++k) r.t0[k] = sea_order_lane(row0 + uint32_t(k * B));

        for (uint32_t i = (p.flags & PF_READ_LIVE) ? 0u : 1u; i < p.n_ops; ++i) {
            const Op& op = p.ops[i];
            if (op.kind == OP_ADVANCE) {
#pragma unroll
                for (int k = 0; k < kJitRows; ++k) r.kill[k] = false;
                jit_run_systems<0>(r, op, __uint_as_float(op.dt_bits), p.adv_frame[i], row0, B);
#pragma unroll
                for (int k = 0; k < kJitRows; ++k) r.m[k] = r.kill[k] ? 0u : r.m[k];  // despawn commands: after the last system
            } else if (op.kind == OP_SAVE) {
                if (!(op.flags & OPF_NO_STORE)) store(p.arena + (size_t(op.image_off256) << 8));
                uint32_t n_alive = 0, bad = 0;
#pragma unroll
                for (int k = 0; k < kJitRows; ++k) n_alive += r.m[k] & 1u;
                unsigned int* a = &s_acc[op.save_index * kAccStride * 2];
                jit_hash_columns<0>(r, a, lane, bad);
                const unsigned full = 0xffffffffu;
                const uint32_t cnt = __reduce_add_sync(full, n_alive);
                const uint32_t anybad = __reduce_or_sync(full, bad);
                if (lane == 0) { atomicAdd(&a[12], cnt); if (anybad) atomicOr(&a[14], 1u); }
            } else {  // OP_LOAD
                load(p.arena + (size_t(op.image_off256) << 8), op.n_rows);
            }
        }
        if (p.flags & PF_WRITE_LIVE_ACTIVE) store(p.arena);
        if (signal_items) {  // every thread's stores of this item are visible at gpu scope, then one release store announces it
            __threadfence();
            __syncthreads();
            if (tid == 0) st_release_gpu(&p.item_done[item], p.done_seq);
        }
        item = next_item;
    }

    // ---- block partials -> global accumulators -> (last block) host-visible results: k_particles_program's protocol ----
    __syncthreads();
    for (uint32_t i = tid; i < p.n_saves * kAccStride; i += B) {
        unsigned long long v = (unsigned long long)s_acc[2 * i] | ((unsigned long long)s_acc[2 * i + 1] << 32);
        const uint32_t c = i % kAccStride;
        if (v) {
            if (c == 6) atomicAdd(&p.accum[i], v);
            else if (c == 7) atomicOr(&p.accum[i], v);
            else atomicXor(&p.accum[i], v);
        }
    }
    __threadfence();
    __syncthreads();
    if (p.trace && tid == 0) atomicMax(&p.trace[1], globaltimer_ns());
    if (tid == 0) s_last = (atomicAdd(p.ticket, 1u) == gridDim.x - 1u);
    __syncthreads();
    if (s_last) {
        __threadfence();
        for (uint32_t i = tid; i < p.n_saves * kAccStride; i += B)
            publish_pair(p.out, i, atomicExch(&p.accum[i], 0ULL), p.seq);
        if (tid == 0) publish_pair(p.out, kSeqIndex, p.seq, p.seq);
        __syncthreads();
        if (tid == 0) {
            p.ticket[0] = 0u;
            p.ticket[1] = 0u;
            if (p.trace) p.trace[2] = globaltimer_ns();
        }
    }
}

}  // namespace bgr
