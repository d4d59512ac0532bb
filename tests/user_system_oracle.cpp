// TEST INFRASTRUCTURE: the oracle's side of user systems (bgr_add_user_system), for CPU-compiled copies of the same source.
//
// The oracle (oracle/world.hpp) runs compiled-in systems only.  This file adds the user-system case on the oracle's own
// World, restating the contract of include/bevy_ggrs_b200.h:
//   * query filter: the system runs on every entity that has every bound column;
//   * the host copy of the source sees typed copies of the elements; only the non-const ones are written back
//     (the trampoline next to the source, tests/user_system_util.py, does that);
//   * bgr_sys_ctx: dt, frame (RollbackFrameCount after the AdvanceWorld increment), n_players / inputs, order
//     (order_base + RollbackOrdered index), params;
//   * cmd.despawn() is deferred with every other despawn command to after the last system of the frame.
// handle_requests / advance_world are World's (world.hpp), restated here only to reach the user-system case; a World made
// here is the oracle's World and every orc_* entry point of liboracle.so works on it.
#include <cstring>
#include <map>
#include <string>
#include <tuple>
#include <utility>

#include "../oracle/world.hpp"
#include "../bevy_ggrs_b200/csrc/user_system.cuh"

using namespace oracle;

#define USR_API extern "C" __attribute__((visibility("default")))

namespace {

// host trampoline of one user system: elems[i] points at the entity's element of bound column i
typedef void (*HostSystemFn)(const bgr_sys_ctx* ctx, uint8_t* const* elems, int* despawn);

constexpr uint32_t kUserBase = 0x1000;  // oracle-side system ids of user systems: kUserBase + index

struct UserSystem {
    HostSystemFn fn;
    std::vector<uint32_t> params;
};
std::map<const World*, std::vector<UserSystem>> g_user;
thread_local std::string g_err;

void run_user_system(World& w, const SystemDesc& s, std::vector<size_t>& despawn) {
    const UserSystem& u = g_user.at(&w).at(s.id - kUserBase);
    bgr_sys_ctx ctx;
    std::memset(&ctx, 0, sizeof ctx);
    ctx.dt = w.ggrs_time.delta_secs;
    ctx.frame = w.rollback_frame_count;
    ctx.n_players = w.n_players;
    std::memcpy(ctx.inputs, w.player_inputs, 8);
    for (size_t j = 0; j < u.params.size() && j < 8; ++j) ctx.params[j] = u.params[j];
    uint8_t* elems[4] = {nullptr, nullptr, nullptr, nullptr};
    for (size_t r = 0; r < w.rows(); ++r) {
        bool has_all = true;
        for (uint32_t c : s.cols) has_all = has_all && w.has[c][r];
        if (!has_all) continue;
        for (size_t i = 0; i < s.cols.size(); ++i) elems[i] = &w.data[s.cols[i]][r * size_t(w.columns[s.cols[i]].elem_bytes)];
        ctx.order = w.order_base + w.rollback_ordered.order_of(w.rollback_id[r]);
        int kill = 0;
        u.fn(&ctx, elems, &kill);
        if (kill) despawn.push_back(r);
    }
}

// World::advance_world (world.hpp) with the user-system case
void advance_world(World& w) {
    uint64_t this_frame = uint64_t(int64_t(w.rollback_frame_count));
    uint64_t runtime = this_frame * 1000000000ULL / uint64_t(w.fps);
    if (runtime < w.ggrs_time.elapsed_ns) throw std::runtime_error("tried to move time backwards");
    w.ggrs_time.delta_ns = runtime - w.ggrs_time.elapsed_ns;
    w.ggrs_time.elapsed_ns = runtime;
    w.ggrs_time.delta_secs = duration_as_secs_f32(w.ggrs_time.delta_ns);
    std::vector<size_t> despawn;
    w.pending_spawns.clear();
    for (const SystemDesc& s : w.systems) {
        if (s.id >= kUserBase) run_user_system(w, s, despawn);
        else w.run_system(s, despawn);
    }
    w.apply_despawns(despawn);
    w.apply_spawns();
}

// World::handle_requests (world.hpp) over the advance_world above
void handle_requests(World& w, const bgr_session_info& sess, const bgr_request* reqs, uint32_t n, std::vector<bgr_checksum>& out) {
    for (uint32_t i = 0; i < n; ++i) {
        const bgr_request& rq = reqs[i];
        int32_t current_frame = w.rollback_frame_count;
        std::optional<uint32_t> maxp;
        std::optional<int32_t> confirmed;
        switch (sess.kind) {
        case BGR_SESSION_P2P: maxp = sess.max_prediction; confirmed = sess.confirmed_frame; break;
        case BGR_SESSION_SYNCTEST: {
            maxp = sess.max_prediction;
            int32_t cf = current_frame - int32_t(sess.check_distance);
            if (cf >= 0) confirmed = cf;
            break;
        }
        case BGR_SESSION_SPECTATOR: maxp = 0; confirmed = current_frame; break;
        default: break;
        }
        if (maxp) w.max_prediction = *maxp;
        if (confirmed) w.confirmed_frame_count = *confirmed;
        switch (rq.kind) {
        case BGR_REQ_SAVE: w.save_world(); out.push_back(bgr_checksum{rq.frame, 1u, w.checksum_lo, 0}); break;
        case BGR_REQ_LOAD: w.rollback_frame_count = rq.frame; w.load_world(); break;
        case BGR_REQ_ADVANCE:
            w.rollback_frame_count += 1;
            w.n_players = rq.n_players;
            std::memcpy(w.player_inputs, rq.inputs, BGR_MAX_PLAYERS);
            advance_world(w);
            w.n_players = 0;
            break;
        default: throw std::runtime_error("bad request kind");
        }
    }
}

template <class F>
int guarded(F&& f) {
    try {
        f();
        return BGR_OK;
    } catch (const RollbackPanic& e) {
        g_err = e.what();
        return BGR_ERR_NO_SNAPSHOT;
    } catch (const NonFinitePanic& e) {
        g_err = e.what();
        return BGR_ERR_NON_FINITE;
    } catch (const std::exception& e) {
        g_err = e.what();
        return BGR_ERR_INVALID_ARGUMENT;
    }
}

}  // namespace

// Invocation glue of a CPU build of a user system: typed copies of the entity's elements, the call, and the write-back of
// the non-const parameters only.  usr_call(&ns::NAME, ...) is what a source's trampoline does.
template <class... A, size_t... I>
void usr_call(void (*fn)(const bgr_sys_ctx&, bgr_commands&, A...), const bgr_sys_ctx* ctx, uint8_t* const* e, int* despawn,
              std::index_sequence<I...>) {
    std::tuple<typename bgr_param<A>::type...> v;
    (std::memcpy(&std::get<I>(v), e[I], sizeof(std::get<I>(v))), ...);
    bgr_commands cmd{false};
    fn(*ctx, cmd, std::get<I>(v)...);
    ((bgr_param<A>::writes ? (void)std::memcpy(e[I], &std::get<I>(v), sizeof(std::get<I>(v))) : (void)0), ...);
    *despawn = cmd.despawn_requested ? 1 : 0;
}
template <class... A>
void usr_call(void (*fn)(const bgr_sys_ctx&, bgr_commands&, A...), const bgr_sys_ctx* ctx, uint8_t* const* e, int* despawn) {
    usr_call(fn, ctx, e, despawn, std::index_sequence_for<A...>{});
}

USR_API const char* usr_last_error() { return g_err.c_str(); }

// orc_add_system for a user system: `fn` is the trampoline of a CPU build of its source
USR_API int usr_add_user_system(World* w, HostSystemFn fn, const uint32_t* cols, uint32_t n_cols, const uint32_t* params, uint32_t n_params) {
    return guarded([&] {
        if (n_cols < 1 || n_cols > 4) throw std::runtime_error("a user system binds 1 to 4 columns");
        std::vector<UserSystem>& us = g_user[w];
        SystemDesc s;
        s.id = kUserBase + uint32_t(us.size());
        s.cols.assign(cols, cols + n_cols);
        us.push_back(UserSystem{fn, std::vector<uint32_t>(params, params + n_params)});
        w->systems.push_back(std::move(s));
    });
}

USR_API void usr_forget_world(World* w) { g_user.erase(w); }

USR_API int usr_advance_world(World* w, const uint8_t* inputs, uint32_t n_players) {
    return guarded([&] {
        w->n_players = n_players;
        std::memset(w->player_inputs, 0, sizeof w->player_inputs);
        if (inputs) std::memcpy(w->player_inputs, inputs, n_players);
        advance_world(*w);
        w->n_players = 0;
    });
}

USR_API int usr_handle_requests(World* w, const bgr_session_info* sess, const bgr_request* reqs, uint32_t n, bgr_checksum* out,
                                uint32_t cap, uint32_t* n_out) {
    std::vector<bgr_checksum> cs;
    int rc = guarded([&] { handle_requests(*w, *sess, reqs, n, cs); });
    uint32_t k = 0;
    for (auto& c : cs) { if (k < cap) out[k] = c; ++k; }
    if (n_out) *n_out = k;
    return rc;
}
