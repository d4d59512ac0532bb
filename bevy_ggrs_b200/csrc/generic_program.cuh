// The one-launch path for ANY registered schema and the compiled GgrsSchedule systems: a whole Vec<GgrsRequest>
// (Load / Advance / Save ...) interpreted by one kernel, like k_particles_program, but without knowing the columns at
// compile time.  One 512-row tile per block iteration lives in SHARED MEMORY for the whole program:
//
//     cp.async.bulk  slot/live image --> shared tile              (LOAD, or the program's first read)
//     ADVANCE : every registered system updates its rows of the shared tile in place (a thread owns its rows for the
//               whole program, so no barrier separates systems; despawn commands are applied after the last system)
//     SAVE    : cp.async.bulk shared tile --> the frame's slot, while all threads hash the checksummed byte ranges
//               of their rows out of the same tile (component_checksum.rs:67-108) and count live rows
//     end     : cp.async.bulk shared tile --> live image
//
// so a SyncTest tick of a box_game / score-and-health style world is ONE launch instead of one launch per request
// and per system (round 1's "stepwise" path, which stays as the fallback for schemas wider than a shared-memory tile).
// Per-entity component presence (BGR_STRATEGY_OPTIONAL) is the row's mask byte: it travels with the tile, and every
// system / checksum applies the reference's query filter per row (kernels.cuh row_matches).
//
// Reference semantics: handle_requests (schedule_systems.rs:170-289) over ComponentSnapshotPlugin::save / load
// (component_snapshot.rs:66-123), the checksum plugins, and the systems listed in include/bevy_ggrs_b200.h.
#pragma once
#ifdef __CUDACC_RTC__  // NVRTC (the engine's run-time specialisation, generic_program_jit.cuh): no host headers
#include "rtc_prelude.cuh"
#else
#include <cuda_runtime.h>
#include <cstdint>
#endif

#ifndef __CUDACC_RTC__
#include "../../include/bevy_ggrs_b200.h"
#endif  // NVRTC: the engine's generated prelude defines the BGR_SYS_* ids (host function declarations cannot be parsed there)
#include "kernels.cuh"
#include "seahash.cuh"
#include "tma_copy.cuh"

namespace bgr {

constexpr int kMaxGenericSys = 8;
// threads per block: 64 / 128 / 256 / 512 = 8 / 4 / 2 / 1 rows of the tile per thread; 128 is the default (four independent
// hash chains interleaved per thread; profiles/r02_generic_block_sweep.txt).  This kernel is the INTERPRETER: it reads the
// schema from its parameter block.  bgr_build also compiles the registration's own kernel with NVRTC when it can
// (generic_program_jit.cuh, jit.hpp), and this one is then only the fallback.

struct SysSpec {
    uint32_t id;      // bgr_system
    uint32_t plane0;  // first word plane the system touches (column's first plane + byte_offset / 4)
    uint32_t plane1;  // second bound column's first plane (Velocity for the Transform/Velocity systems)
    uint32_t need;    // absent bits of the bound columns: the query matches a row iff row_matches(mask, need)
    uint32_t param;   // k (U32_ADD / U32_SATSUB_DESPAWN) or the system's index among the call-count systems
};

struct GenericParams {
    uint8_t* arena;
    unsigned long long order_base;
    unsigned long long* accum;  // device [kMaxSaves][kAccStride]
    unsigned long long* out;    // host-mapped result block (same layout / protocol as k_particles_program)
    unsigned int* ticket;       // [0] block-completion ticket, [1] dynamic tile counter
    unsigned long long seq;
    unsigned long long* trace;
    uint32_t words, tile_bytes, n_ops, n_saves, n_tiles, live_rows, flags, n_hash, n_sys;
    // overlap of consecutive launches (generated kernel only; the protocol of k_particles_program's PF_TILE_SIGNAL / PF_TILE_WAIT
    // per WORK ITEM): item_done[i] = sequence number of the last signalling launch whose stores of item i are visible
    unsigned int* item_done;
    uint32_t done_seq, wait_seq, wait_items;
    HashSpec hash[kMaxHashCols];
    SysSpec sys[kMaxGenericSys];
    Op ops[kMaxOps];
    int32_t adv_frame[kMaxOps];  // ADVANCE: RollbackFrameCount after the frame's increment (user systems' bgr_sys_ctx::frame)
};
static_assert(sizeof(GenericParams) <= 4000, "kernel parameter block must fit 4 KB");

// seahash of bytes [off, off+len) of one row's element whose words are `col[w * kTileRows]` (a column of the shared tile)
// (__noinline__: inlined per checksummed column and per row the interpreter grew to 11k instructions — 176 KB of code,
// more than the SM's instruction cache — and ran 2.7x slower per frame than the specialised bundle kernel)
__device__ __noinline__ uint64_t hash_row_range(const uint32_t* col, uint32_t off, uint32_t len) {
    if (((off | len) & 3u) == 0u) {  // word-aligned range (every POD of u32 / f32 / u64 fields): no byte shuffling
        const uint32_t* w = col + size_t(off >> 2) * kTileRows;
        // the common element sizes without a loop (warp-uniform switch: every row of a column has the same range)
        switch (len) {
        case 4: return sea_diffuse(sea_diffuse(kSeaA ^ uint64_t(w[0])) ^ kSeaB ^ kSeaC ^ kSeaD ^ 4ULL);
        case 8: return sea_hash_u64(uint64_t(w[0]) | (uint64_t(w[kTileRows]) << 32));
        case 12: return sea_hash_12(uint64_t(w[0]) | (uint64_t(w[kTileRows]) << 32), w[2 * kTileRows]);
        case 16: return sea_hash_2xu64(uint64_t(w[0]) | (uint64_t(w[kTileRows]) << 32), uint64_t(w[2 * kTileRows]) | (uint64_t(w[3 * kTileRows]) << 32));
        default: break;
        }
        uint64_t a = kSeaA, b = kSeaB, c = kSeaC, d = kSeaD;
        uint32_t i = 0;
        for (; i + 8 <= len; i += 8) {
            const uint64_t x = uint64_t(w[0]) | (uint64_t(w[kTileRows]) << 32);
            w += 2 * kTileRows;
            const uint64_t t = sea_diffuse(a ^ x);
            a = b; b = c; c = d; d = t;
        }
        if (i < len) a = sea_diffuse(a ^ uint64_t(w[0]));
        return sea_diffuse(a ^ b ^ c ^ d ^ uint64_t(len));
    }
    auto byte_at = [&](uint32_t q) -> uint8_t {
        const uint32_t bb = off + q;
        return uint8_t(col[size_t(bb >> 2) * kTileRows] >> (8 * (bb & 3u)));
    };
    return sea_hash_stream(len, byte_at);
}

// One checksummed column whose element is NW whole words (4 * NW bytes, word-aligned) for the thread's R rows:
// `col` points at the first word of the thread's first row, rows are `B` words apart, words of an element kTileRows apart.
// Branch-free per row (a row without the component contributes 0), so the rows' hash chains interleave.
template <int NW, int R, int B>
__device__ __forceinline__ void hash_words_column(const uint32_t* col, const uint32_t (&m)[R], uint32_t absent, uint32_t finite,
                                                  const uint64_t (&t0)[R], uint64_t& hx, uint32_t& bad) {
#pragma unroll
    for (int k = 0; k < R; ++k) {
        uint32_t w[NW];
#pragma unroll
        for (int j = 0; j < NW; ++j) w[j] = col[k * B + j * kTileRows];
        const bool has = row_matches(m[k], absent);  // Query<(&RollbackId, &T)>: exists and has the component
        uint32_t nonfinite = 0;
#pragma unroll
        for (int j = 0; j < NW; ++j) nonfinite |= f32_bits_nonfinite(w[j]);
        bad |= (has && finite) ? nonfinite : 0u;
        uint64_t h;
        if (NW == 1) h = sea_diffuse(sea_diffuse(kSeaA ^ uint64_t(w[0])) ^ kSeaB ^ kSeaC ^ kSeaD ^ 4ULL);
        else if (NW == 2) h = sea_hash_u64(uint64_t(w[0]) | (uint64_t(w[1 % NW]) << 32));
        else if (NW == 3) h = sea_hash_12(uint64_t(w[0]) | (uint64_t(w[1 % NW]) << 32), w[2 % NW]);
        else h = sea_hash_2xu64(uint64_t(w[0]) | (uint64_t(w[1 % NW]) << 32), uint64_t(w[2 % NW]) | (uint64_t(w[3 % NW]) << 32));
        const uint64_t e = sea_hash_entity(t0[k], h);
        hx ^= has ? e : 0ULL;
    }
}

template <int kGenericBlock>
__global__ void __launch_bounds__(kGenericBlock) k_generic_program(const __grid_constant__ GenericParams p) {
    constexpr int kRows = kTileRows / kGenericBlock;  // rows of a tile per thread
    extern __shared__ __align__(128) uint8_t s_buf[];  // one tile
    __shared__ unsigned int s_acc[kMaxSaves * kAccStride * 2];
    __shared__ __align__(8) uint64_t s_bar;
    __shared__ uint32_t s_next;
    __shared__ unsigned int s_last;

    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    if (p.trace && tid == 0) atomicMin(&p.trace[0], globaltimer_ns());
    for (uint32_t i = tid; i < p.n_saves * kAccStride * 2; i += kGenericBlock) s_acc[i] = 0u;
    if (tid == 0) { mbar_init(&s_bar, 1); fence_mbar_init(); }
    __syncthreads();

    // ONE tile buffer.  (A ping-pong pair — ADVANCE reading one buffer and writing the other so that a SAVE's bulk store
    // could keep reading — was measured: no faster, the store has long finished reading when the next ADVANCE starts,
    // and it costs a copy of every word per frame and half the resident blocks.)
    uint8_t* const s_tile = s_buf;
    uint8_t* const s_alive = s_tile + size_t(p.words) * kPlaneBytes;
    uint32_t* const tile_w = reinterpret_cast<uint32_t*>(s_tile);  // word (plane, row) = tile_w[plane * kTileRows + row]
    uint32_t phase = 0;
    bool store_pending = false;  // a bulk store may still be reading the shared tile (block-uniform)

    // the shared tile is about to be modified: pending bulk stores must have read it
    auto before_write = [&]() {
        if (store_pending) {
            if (tid == 0) tma_wait_read<0>();
            __syncthreads();
            store_pending = false;
        }
    };
    // bring tile `t` of image `img` into shared memory; rows the image never contained come back dead
    auto load_tile = [&](const uint8_t* img, uint32_t t, uint32_t n_rows_src) {
        __syncthreads();  // every thread is done with the previous content
        if (tid == 0) {
            tma_wait_read<0>();
            mbar_arrive_expect_tx(&s_bar, p.tile_bytes);
            tma_load_1d(s_tile, img + size_t(t) * p.tile_bytes, p.tile_bytes, &s_bar);
        }
        mbar_wait(&s_bar, phase);
        phase ^= 1u;
        store_pending = false;
        if (size_t(t + 1) * kTileRows > n_rows_src) {
#pragma unroll
            for (int k = 0; k < kRows; ++k) {
                const uint32_t r = tid + k * kGenericBlock;
                if (t * kTileRows + r >= n_rows_src) s_alive[r] = 0;
            }
        }
    };
    auto store_tile = [&](uint8_t* img, uint32_t t) {
        fence_proxy_async();  // generic-proxy writes of this thread are visible to the bulk (async-proxy) store
        __syncthreads();
        if (tid == 0) {
            tma_store_1d(img + size_t(t) * p.tile_bytes, s_tile, p.tile_bytes);
            tma_commit();
        }
        store_pending = true;
    };

    const uint8_t* first_img = p.arena + ((p.flags & PF_READ_LIVE) ? size_t(0) : (size_t(p.ops[0].image_off256) << 8));
    const uint32_t first_rows = (p.flags & PF_READ_LIVE) ? p.live_rows : p.ops[0].n_rows;

    for (uint32_t tile = blockIdx.x; tile < p.n_tiles;) {
        __syncthreads();  // every thread has read the previous s_next
        if (tid == 0) s_next = gridDim.x + atomicAdd(&p.ticket[1], 1u);  // the block's next tile (read after the barrier in load_tile)
        load_tile(first_img, tile, first_rows);
        const uint32_t next_tile = s_next;
        // first lane of the per-entity hash: only depends on the RollbackOrdered index — once per tile, not per SAVE
        const unsigned long long row0 = p.order_base + size_t(tile) * kTileRows + tid;
        uint64_t t0[kRows];
#pragma unroll
        for (int k = 0; k < kRows; ++k) t0[k] = sea_order_lane(row0 + uint32_t(k * kGenericBlock));

        for (uint32_t i = (p.flags & PF_READ_LIVE) ? 0u : 1u; i < p.n_ops; ++i) {
            const Op& op = p.ops[i];
            if (op.kind == OP_ADVANCE) {
                before_write();
                const float dt = __uint_as_float(op.dt_bits);
                // systems outside, the thread's rows inside: a system's spec is decoded once for all of them.  A row still
                // sees the schedule's systems in order, every system sees the entity's presence as it was before the frame,
                // and despawn commands are applied after the last system.
                uint32_t m[kRows];
                bool kill[kRows];
#pragma unroll
                for (int k = 0; k < kRows; ++k) { m[k] = s_alive[tid + k * kGenericBlock]; kill[k] = false; }
#pragma unroll 1
                for (uint32_t s = 0; s < p.n_sys; ++s) {
                    const SysSpec sy = p.sys[s];
                    uint32_t* w0 = tile_w + sy.plane0 * uint32_t(kTileRows) + tid;
                    switch (sy.id) {
                    case BGR_SYS_U32_ADD:
#pragma unroll
                        for (int k = 0; k < kRows; ++k)
                            if (row_matches(m[k], sy.need)) w0[k * kGenericBlock] += sy.param;
                        break;
                    case BGR_SYS_U32_SATSUB_DESPAWN:
#pragma unroll
                        for (int k = 0; k < kRows; ++k)
                            if (row_matches(m[k], sy.need)) {
                                uint32_t v = w0[k * kGenericBlock];
                                v = v > sy.param ? v - sy.param : 0u;
                                w0[k * kGenericBlock] = v;
                                kill[k] = kill[k] || v == 0u;
                            }
                        break;
                    case BGR_SYS_U32_STORE_CALL_COUNT:
#pragma unroll
                        for (int k = 0; k < kRows; ++k)
                            if (row_matches(m[k], sy.need)) w0[k * kGenericBlock] = op.call_count + sy.param;
                        break;
                    case BGR_SYS_DESPAWN_ON_INPUT: {  // param = player handle | value << 8
                        const uint32_t player = sy.param & 0xFFu, n_players = (op.flags >> 8) & 0xFu;
                        const uint32_t input = player < n_players && player < 8 ? op.inputs[player] : 0u;
                        const bool hit = input == (sy.param >> 8);
#pragma unroll
                        for (int k = 0; k < kRows; ++k) kill[k] = kill[k] || (hit && row_matches(m[k], sy.need));
                        break;
                    }
                    case BGR_SYS_PARTICLES_UPDATE: {
                        uint32_t* v0 = tile_w + sy.plane1 * uint32_t(kTileRows) + tid;
#pragma unroll
                        for (int k = 0; k < kRows; ++k)
                            if (row_matches(m[k], sy.need)) {
                                uint32_t* t = w0 + k * kGenericBlock;
                                uint32_t* v = v0 + k * kGenericBlock;
                                uint32_t tx = t[0], ty = t[kTileRows], tz = t[2 * kTileRows], vx = v[0], vy = v[kTileRows], vz = v[2 * kTileRows];
                                particle_step(tx, ty, tz, vx, vy, vz, dt);
                                t[0] = tx; t[kTileRows] = ty; t[2 * kTileRows] = tz; v[0] = vx; v[kTileRows] = vy; v[2 * kTileRows] = vz;
                            }
                        break;
                    }
                    case BGR_SYS_PARTICLES_DESPAWN:
#pragma unroll
                        for (int k = 0; k < kRows; ++k)
                            if (row_matches(m[k], sy.need)) {
                                uint32_t* t = w0 + k * kGenericBlock;
                                uint64_t ttl = (uint64_t(t[kTileRows]) << 32) | t[0];
                                ttl -= 1;
                                t[0] = uint32_t(ttl); t[kTileRows] = uint32_t(ttl >> 32);
                                kill[k] = kill[k] || ttl == 0;
                            }
                        break;
                    case BGR_SYS_BOX_MOVE: {
                        uint32_t* v0 = tile_w + sy.plane1 * uint32_t(kTileRows) + tid;
                        const uint32_t n_players = (op.flags >> 8) & 0xFu;
#pragma unroll
                        for (int k = 0; k < kRows; ++k)
                            if (row_matches(m[k], sy.need)) {
                                float* t = reinterpret_cast<float*>(w0 + k * kGenericBlock);
                                float* v = reinterpret_cast<float*>(v0 + k * kGenericBlock);
                                float tx = t[0], ty = t[kTileRows], tz = t[2 * kTileRows], vx = v[0], vy = v[kTileRows], vz = v[2 * kTileRows];
                                const unsigned long long handle = row0 + uint32_t(k * kGenericBlock);
                                const uint32_t input = handle < n_players && handle < 8 ? op.inputs[handle] : 0u;
                                box_move_step(tx, ty, tz, vx, vy, vz, dt, input);
                                t[0] = tx; t[kTileRows] = ty; t[2 * kTileRows] = tz; v[0] = vx; v[kTileRows] = vy; v[2 * kTileRows] = vz;
                            }
                        break;
                    }
                    default: break;
                    }
                }
#pragma unroll
                for (int k = 0; k < kRows; ++k)
                    if (kill[k]) s_alive[tid + k * kGenericBlock] = 0;
            } else if (op.kind == OP_SAVE) {
                // the bulk store streams the tile to the frame's slot while the threads hash their rows out of it
                if (!(op.flags & OPF_NO_STORE)) store_tile(p.arena + (size_t(op.image_off256) << 8), tile);
                uint32_t m[kRows];
                uint32_t n_alive = 0, bad = 0;
#pragma unroll
                for (int k = 0; k < kRows; ++k) {
                    m[k] = s_alive[tid + k * kGenericBlock];
                    n_alive += m[k] & 1u;
                }
                const unsigned full = 0xffffffffu;
                unsigned int* a = &s_acc[op.save_index * kAccStride * 2];
#pragma unroll 1
                for (uint32_t c = 0; c < p.n_hash; ++c) {  // one checksummed column at a time
                    const HashSpec hs = p.hash[c];
                    const uint32_t* col = tile_w + (hs.first_plane + (hs.off >> 2)) * uint32_t(kTileRows) + tid;
                    uint64_t hx = 0;
                    // the common element shapes (whole u32 / f32 / u64 fields, 4..16 bytes) inline and branch-free per
                    // row; anything else through the one out-of-line copy of the general hash.  The switch is uniform.
                    const uint32_t shape = ((hs.off | hs.len) & 3u) == 0u ? hs.len >> 2 : 0u;
                    switch (shape) {
                    case 1: hash_words_column<1, kRows, kGenericBlock>(col, m, hs.absent, hs.finite, t0, hx, bad); break;
                    case 2: hash_words_column<2, kRows, kGenericBlock>(col, m, hs.absent, hs.finite, t0, hx, bad); break;
                    case 3: hash_words_column<3, kRows, kGenericBlock>(col, m, hs.absent, hs.finite, t0, hx, bad); break;
                    case 4: hash_words_column<4, kRows, kGenericBlock>(col, m, hs.absent, hs.finite, t0, hx, bad); break;
                    default: {
                        const uint32_t* base = tile_w + hs.first_plane * uint32_t(kTileRows) + tid;
#pragma unroll
                        for (int k = 0; k < kRows; ++k) {
                            if (!row_matches(m[k], hs.absent)) continue;  // Query<(&RollbackId, &T)>: exists and has the component
                            if (hs.finite)
                                for (uint32_t q = 0; q + 4 <= hs.len; q += 4) bad |= f32_bits_nonfinite(base[k * kGenericBlock + ((hs.off + q) >> 2) * uint32_t(kTileRows)]);
                            hx ^= sea_hash_entity(t0[k], hash_row_range(base + k * kGenericBlock, hs.off, hs.len));
                        }
                    }
                    }
                    const uint32_t lo = __reduce_xor_sync(full, uint32_t(hx)), hi = __reduce_xor_sync(full, uint32_t(hx >> 32));
                    if (lane == 0) { atomicXor(&a[2 * hs.slot], lo); atomicXor(&a[2 * hs.slot + 1], hi); }
                }
                const uint32_t cnt = __reduce_add_sync(full, n_alive);
                const uint32_t anybad = __reduce_or_sync(full, bad);
                if (lane == 0) { atomicAdd(&a[12], cnt); if (anybad) atomicOr(&a[14], 1u); }
            } else {  // OP_LOAD
                load_tile(p.arena + (size_t(op.image_off256) << 8), tile, op.n_rows);
            }
        }
        if (p.flags & PF_WRITE_LIVE_ACTIVE) store_tile(p.arena, tile);
        tile = next_tile;
    }
    if (tid == 0) tma_wait_all();  // every bulk store has landed before the results are published

    // ---- block partials -> global accumulators -> (last block) host-visible results: k_particles_program's protocol ----
    __syncthreads();
    for (uint32_t i = tid; i < p.n_saves * kAccStride; i += kGenericBlock) {
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
        for (uint32_t i = tid; i < p.n_saves * kAccStride; i += kGenericBlock)
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
