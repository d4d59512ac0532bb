// C++ host-side mirror of the bevy_ggrs plugin surface for the rollback hot path, above the C ABI
// (include/bevy_ggrs_b200.h).  Same names, argument meaning and error behaviour as the reference:
//
//   App app(max_entities, max_depth);
//   app.add_plugins(GgrsPlugin<GgrsConfig<uint8_t>>{})                 // lib.rs:198-258
//      .insert_resource(RollbackFrameRate{60})                         // time.rs:19-26
//      .add_systems(ReadInputs{}, read_local_inputs)                   // lib.rs:148-149
//      .rollback_component_with_clone<Transform>()                     // rollback_app.rs:178-183
//      .rollback_component_with_copy<Velocity>()                       // rollback_app.rs:157-162
//      .checksum_component<Transform>(hash_bytes(0, 12, true))         // rollback_app.rs:227-232
//      .add_systems(GgrsSchedule{}, System{BGR_SYS_PARTICLES_UPDATE, {col<Transform>, col<Velocity>}})
//      .insert_resource(Session::SyncTest(ggrs::SyncTestSession(2, 8, 9, 2)))
//      .add_observer([](const SyncTestMismatch& m) { ... });
//   app.update();                                                      // run_ggrs_schedules, schedule_systems.rs:19-83
//
// A Rust panic becomes a C++ exception carrying the same text (`Panic`).  The "World" is the engine:
// columns and the snapshot ring live in HBM, this layer holds no component data.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <typeindex>
#include <typeinfo>
#include <vector>

#include "../../include/bevy_ggrs_b200.h"
#include "ggrs_standin.hpp"

namespace bevy_ggrs {

struct Panic : std::runtime_error {
    int status;
    Panic(int s, const std::string& text) : std::runtime_error(text), status(s) {}
};
inline void check(int status) {
    if (status != BGR_OK) throw Panic(status, bgr_last_error());
}

// ---- schedule labels / resources / events (lib.rs:73-149, snapshot/mod.rs:66-77) ----
struct GgrsSchedule {};
struct ReadInputs {};
struct Startup {};
struct RollbackFrameRate { size_t fps = 60; };
struct LocalPlayers { std::vector<ggrs::PlayerHandle> handles; };
struct LocalInputs { std::map<ggrs::PlayerHandle, uint8_t> inputs; };
struct SyncTestMismatch { ggrs::Frame current_frame; std::vector<ggrs::Frame> mismatched_frames; };
template <class Input = uint8_t> struct GgrsConfig { using input_type = Input; };
template <class Config> struct GgrsPlugin {};

struct Session {  // lib.rs:79-86: enum Session<T> { SyncTest(..), P2P(..), Spectator(..) }
    enum Kind { SyncTestKind, P2PKind, SpectatorKind } kind = SyncTestKind;
    std::shared_ptr<ggrs::SyncTestSession> synctest;
    std::shared_ptr<ggrs::P2PTraceSession> p2p;
    std::shared_ptr<ggrs::SpectatorTraceSession> spectator;
    static Session SyncTest(ggrs::SyncTestSession s) { Session r; r.kind = SyncTestKind; r.synctest = std::make_shared<ggrs::SyncTestSession>(std::move(s)); return r; }
    static Session P2P(ggrs::P2PTraceSession s) { Session r; r.kind = P2PKind; r.p2p = std::make_shared<ggrs::P2PTraceSession>(std::move(s)); return r; }
    static Session Spectator(ggrs::SpectatorTraceSession s) { Session r; r.kind = SpectatorKind; r.spectator = std::make_shared<ggrs::SpectatorTraceSession>(std::move(s)); return r; }
};

// a compiled-in GgrsSchedule system: id + bound columns + scalar parameters
struct System {
    uint32_t id;
    std::vector<uint32_t> columns;
    std::vector<uint32_t> params;
};
// A GgrsSchedule system of the game's own, as CUDA source (bgr_add_user_system: the contract is in the header).
struct CudaSystem {
    std::string name, source;
    std::vector<uint32_t> columns;
    std::vector<uint32_t> params;
};

// A GgrsSchedule system that only touches host-side resources (box_game.rs:146-148 increase_frame_system).
// Resources are a few bytes and not data-parallel: they stay on the host, this layer rolls them back per frame
// (resource_snapshot.rs:65-93) and XORs their checksum parts into the engine's checksum (checksum.rs:88-99).
class App;
struct ResourceSystem { std::function<void(App&)> fn; };

// what a `fn(&T) -> u64` hasher becomes across the C ABI: seahash of a byte range of the element
struct ByteRangeHasher { uint32_t offset, len; bool assert_finite; };
inline ByteRangeHasher hash_bytes(uint32_t offset, uint32_t len, bool assert_finite = false) { return {offset, len, assert_finite}; }

class App {
public:
    App(uint32_t max_entities, uint32_t max_depth, int device = 0, uint32_t flags = 0) {
        bgr_config cfg;
        std::memset(&cfg, 0, sizeof cfg);
        cfg.abi_version = BGR_ABI_VERSION; cfg.device = device; cfg.max_entities = max_entities;
        cfg.max_depth = max_depth; cfg.fps = 60; cfg.flags = flags;
        cfg_ = cfg;
    }
    ~App() { if (engine_) bgr_engine_destroy(engine_); }
    App(const App&) = delete;

    template <class C> App& add_plugins(GgrsPlugin<C>) { return *this; }
    App& insert_resource(RollbackFrameRate r) { cfg_.fps = uint32_t(r.fps); return *this; }
    App& insert_resource(Session s) { session_ = std::move(s); return *this; }
    App& remove_session() { session_.reset(); return *this; }  // world.remove_resource::<Session<T>>()
    App& insert_resource(LocalInputs li) { local_inputs_ = std::move(li); return *this; }
    App& add_systems(ReadInputs, std::function<void(App&)> f) { read_inputs_.push_back(std::move(f)); return *this; }
    App& add_systems(Startup, std::function<void(App&)> f) { startup_.push_back(std::move(f)); return *this; }
    App& add_systems(GgrsSchedule, System s) { systems_.push_back(std::move(s)); cuda_systems_.emplace_back(); return *this; }
    App& add_systems(GgrsSchedule, CudaSystem s) { systems_.push_back(System{}); cuda_systems_.push_back(std::move(s)); return *this; }
    App& add_systems(GgrsSchedule, ResourceSystem s) { res_systems_.push_back(std::move(s.fn)); return *this; }
    App& add_observer(std::function<void(const SyncTestMismatch&)> f) { observers_.push_back(std::move(f)); return *this; }

    // ---- RollbackApp (rollback_app.rs:31-248) ----
    template <class T> App& rollback_component_with_copy() { return register_component<T>(BGR_STRATEGY_COPY); }
    // Clone of plain bytes -> an HBM column.  Clone of anything else (bevy's Sprite holds an Arc asset handle,
    // particles.rs:191) -> the type stays on the host in a side table keyed by row (= RollbackOrdered index, never
    // reused) and is rolled back there by the same request vectors: Save clones the table into a per-frame snapshot
    // (component_snapshot.rs:66-90), Load replaces it by a clone of the frame's snapshot = the four-way match of
    // component_snapshot.rs:99-115 for every entity at once; whether the entity exists is the alive mask in HBM.
    template <class T> App& rollback_component_with_clone() {
        if constexpr (std::is_trivially_copyable<T>::value) return register_component<T>(BGR_STRATEGY_CLONE);
        else { host_cols_[std::type_index(typeid(T))] = std::make_unique<HostColumn<T>>(); return *this; }
    }
    // commands.entity(row).insert(value) / .remove::<T>() / Query<&T> for a host-side component
    template <class T> void host_insert(uint32_t row, T value) {
        if (!entity_exists(row)) throw Panic(BGR_ERR_INVALID_ARGUMENT, "entity of row " + std::to_string(row) + " does not exist");
        host_col<T>().live.insert_or_assign(row, std::move(value));
    }
    template <class T> void host_remove(uint32_t row) { host_col<T>().live.erase(row); }
    template <class T> const T* host_get(uint32_t row) {
        auto& live = host_col<T>().live;
        auto it = live.find(row);
        return it != live.end() && entity_exists(row) ? &it->second : nullptr;
    }
    template <class T> std::vector<ggrs::Frame> host_snapshot_frames() {
        std::vector<ggrs::Frame> f;
        for (auto& kv : host_col<T>().snaps) f.push_back(kv.first);
        return f;
    }
    // a component single entities may lose / regain inside the window: Option<&mut T> in ComponentSnapshotPlugin::load
    // (component_snapshot.rs:99-115); see remove<T>() / insert<T>() below
    template <class T> App& rollback_optional_component_with_copy() { return register_component<T>(BGR_STRATEGY_COPY | BGR_STRATEGY_OPTIONAL); }
    template <class T> App& rollback_optional_component_with_clone() { return register_component<T>(BGR_STRATEGY_CLONE | BGR_STRATEGY_OPTIONAL); }
    template <class T> App& checksum_component(ByteRangeHasher h) { checksums_.push_back({col<T>(), h}); return *this; }
    template <class T> App& checksum_component_with_hash() { return checksum_component<T>(hash_bytes(0, uint32_t(sizeof(T)))); }

    // rollback_resource_with_copy / _with_clone (rollback_app.rs:171-176, 192-197) and
    // checksum_resource_with_hash (rollback_app.rs:213-218) for POD resources, host-side
    template <class R> App& rollback_resource_with_copy(const R& initial) {
        static_assert(std::is_trivially_copyable<R>::value, "POD resources only");
        std::vector<uint8_t> b(sizeof(R));
        std::memcpy(b.data(), &initial, sizeof(R));
        resources_[std::type_index(typeid(R))] = std::move(b);
        return *this;
    }
    template <class R> App& rollback_resource_with_clone(const R& initial) { return rollback_resource_with_copy<R>(initial); }
    template <class R> App& checksum_resource_with_hash() { res_checksummed_.push_back(std::type_index(typeid(R))); return *this; }
    template <class R> R& resource() {
        auto it = resources_.find(std::type_index(typeid(R)));
        if (it == resources_.end()) throw Panic(BGR_ERR_MISSING_RESOURCE, std::string("Requested resource does not exist: ") + typeid(R).name());
        return *reinterpret_cast<R*>(it->second.data());
    }

    template <class T> uint32_t col() const {
        auto it = columns_.find(std::type_index(typeid(T)));
        if (it == columns_.end()) throw Panic(BGR_ERR_INVALID_ARGUMENT, std::string("component not registered for rollback: ") + typeid(T).name());
        return it->second;
    }

    // ---- World access ----
    const LocalPlayers& local_players() const { return local_players_; }
    uint32_t spawn(uint32_t count) { finish(); uint32_t first = 0; check(bgr_spawn(engine_, count, &first)); return first; }
    template <class T> void write(uint32_t first_row, const std::vector<T>& v) {
        finish();
        check(bgr_write_component(engine_, col<T>(), first_row, uint32_t(v.size()), v.data(), uint32_t(sizeof(T))));
    }
    template <class T> std::vector<T> read(uint32_t first_row, uint32_t count) {
        std::vector<T> v(count);
        check(bgr_read_component(engine_, col<T>(), first_row, count, v.data(), uint32_t(sizeof(T))));
        return v;
    }
    // commands.entity(row).remove::<T>() / .insert(value) / Query<Has<T>> for optional components
    template <class T> void remove(uint32_t row) { finish(); check(bgr_remove_component(engine_, col<T>(), row)); }
    template <class T> void insert(uint32_t row, const T& value) { finish(); check(bgr_insert_component(engine_, col<T>(), row, &value)); }
    template <class T> std::vector<uint8_t> has(uint32_t first_row, uint32_t count) {
        std::vector<uint8_t> v(count);
        check(bgr_has_component(engine_, col<T>(), first_row, count, v.data()));
        return v;
    }
    // asynchronous host mirror of bytes [offset, offset+len) of every T in rows [first_row, first_row+count):
    // `dst` from bgr_host_alloc; readable after download_wait(ticket)
    template <class T> uint32_t download_begin(uint32_t offset, uint32_t len, uint32_t first_row, uint32_t count, void* dst) {
        uint32_t ticket = 0;
        check(bgr_download_begin(engine_, col<T>(), offset, len, first_row, count, dst, &ticket));
        return ticket;
    }
    void download_wait(uint32_t ticket) { check(bgr_download_wait(engine_, ticket)); }
    // GgrsComponentSnapshots<T>::peek(frame) (mod.rs:233-240)
    template <class T> std::optional<std::vector<T>> peek(ggrs::Frame frame, uint32_t first_row, uint32_t count) {
        std::vector<T> v(count);
        int32_t found = 0;
        check(bgr_peek(engine_, frame, col<T>(), first_row, count, v.data(), uint32_t(sizeof(T)), nullptr, &found));
        if (!found) return std::nullopt;
        return v;
    }
    uint64_t active_count() { uint64_t n = 0; check(bgr_active_count(engine_, &n)); return n; }
    int32_t rollback_frame_count() { int32_t f = 0; check(bgr_rollback_frame_count(engine_, &f)); return f; }
    int32_t confirmed_frame_count() { int32_t f = 0; check(bgr_confirmed_frame_count(engine_, &f)); return f; }
    uint64_t launch_count() { uint64_t n = 0; check(bgr_launch_count(engine_, &n)); return n; }
    bgr_engine* engine() { finish(); return engine_; }
    const std::vector<bgr_checksum>& last_checksums() const { return last_checksums_; }

    // ---- one Bevy frame: run_ggrs_schedules (schedule_systems.rs:19-83) ----
    void update() {
        finish();
        // bevy Time<Real>: zero delta on the first update, then TimeUpdateStrategy::ManualDuration(1/60 s)
        const uint64_t delta = first_update_ ? 0 : 16666667ull;
        first_update_ = false;
        const uint64_t fps_delta = run_slow_ ? 1000000000ull * 11 / (uint64_t(cfg_.fps) * 10) : 1000000000ull / cfg_.fps;
        accumulator_ns_ += delta;
        if (session_ && session_->kind == Session::P2PKind) session_->p2p->poll_remote_clients();             // :43-53
        if (session_ && session_->kind == Session::SpectatorKind) session_->spectator->poll_remote_clients();
        while (accumulator_ns_ >= fps_delta) {
            accumulator_ns_ -= fps_delta;
            if (!session_) {  // :70-79 "No session has been started yet, reset time data and snapshots"
                accumulator_ns_ = 0; run_slow_ = false;
                local_players_.handles.clear();
                check(bgr_reset_session(engine_));  // RollbackFrameCount(0), ConfirmedFrameCount(-1), MaxPredictionWindow(8)
                return;
            }
            tick();
        }
    }
    // exactly one GGRS tick (benches)
    void step() { finish(); tick(); }
    uint32_t max_prediction_window() { uint32_t v = 0; check(bgr_max_prediction_window(engine_, &v)); return v; }
    std::vector<int32_t> snapshot_frames() {
        int32_t f[128]; uint32_t n = 0;
        check(bgr_snapshot_frames(engine_, f, 128, &n));
        return std::vector<int32_t>(f, f + std::min<uint32_t>(n, 128));
    }

private:
    template <class T> App& register_component(uint32_t strategy) {
        static_assert(std::is_trivially_copyable<T>::value, "only POD components cross the C ABI");
        pending_cols_.push_back({std::type_index(typeid(T)), typeid(T).name(), uint32_t(sizeof(T)), strategy});
        columns_[std::type_index(typeid(T))] = uint32_t(pending_cols_.size() - 1);
        return *this;
    }
    void finish() {  // end of App::build
        if (engine_) return;
        check(bgr_engine_create(&cfg_, &engine_));
        for (auto& c : pending_cols_) { uint32_t id = 0; check(bgr_rollback_component(engine_, c.name.c_str(), c.bytes, c.strategy, &id)); }
        for (auto& ck : checksums_)
            check(bgr_checksum_component(engine_, ck.first, BGR_HASH_BYTES, ck.second.offset, ck.second.len,
                                         ck.second.assert_finite ? BGR_HASH_FLAG_ASSERT_FINITE_F32 : 0u));
        for (size_t i = 0; i < systems_.size(); ++i) {  // add_systems order, compiled-in and user systems interleaved
            const System& s = systems_[i];
            const CudaSystem& u = cuda_systems_[i];
            if (!u.name.empty())
                check(bgr_add_user_system(engine_, u.name.c_str(), u.source.c_str(), u.columns.data(), uint32_t(u.columns.size()),
                                          u.params.data(), uint32_t(u.params.size())));
            else
                check(bgr_add_system(engine_, s.id, s.columns.data(), uint32_t(s.columns.size()), s.params.data(), uint32_t(s.params.size())));
        }
        check(bgr_build(engine_));
        for (auto& f : startup_) f(*this);
    }

    void tick() {  // :59-69: depending on the session type, doing a single update looks a bit different
        switch (session_->kind) {
        case Session::SyncTestKind: run_synctest(*session_->synctest); break;
        case Session::P2PKind: run_slow_ = session_->p2p->frames_ahead() > 0; run_p2p(*session_->p2p); break;
        case Session::SpectatorKind: run_spectator(*session_->spectator); break;
        }
    }

    // run_p2p (schedule_systems.rs:137-168)
    void run_p2p(ggrs::P2PTraceSession& sess) {
        local_players_.handles = sess.local_player_handles();
        if (sess.current_state() != ggrs::SessionState::Running) return;
        local_inputs_.reset();
        for (auto& f : read_inputs_) f(*this);
        if (!local_inputs_)
            throw Panic(BGR_ERR_MISSING_RESOURCE, "No local player inputs found. Did you insert systems into the ReadInputs schedule?");
        for (auto& kv : local_inputs_->inputs) sess.add_local_input(kv.first, kv.second);
        const auto requests = sess.advance_frame();
        // the numbers handle_requests reads from a P2P session before every request (:203-206)
        bgr_session_info info{BGR_SESSION_P2P, uint32_t(sess.max_prediction()), 0, sess.confirmed_frame()};
        handle_requests(requests, info, [&](ggrs::Frame f, unsigned __int128 c) { sess.save_cell(f, c); });
    }

    // run_spectator (schedule_systems.rs:120-135): only AdvanceFrame requests, several per tick when catching up
    void run_spectator(ggrs::SpectatorTraceSession& sess) {
        if (sess.current_state() != ggrs::SessionState::Running) return;
        const auto requests = sess.advance_frame();
        if (requests.empty()) return;  // PredictionThreshold: "Waiting for input from host."
        bgr_session_info info{BGR_SESSION_SPECTATOR, 0, 0, 0};  // max_prediction forced to 0, confirmed = current frame (:199-201, :209)
        handle_requests(requests, info, [](ggrs::Frame, unsigned __int128) {});
    }

    // run_synctest (schedule_systems.rs:85-118)
    void run_synctest(ggrs::SyncTestSession& sess) {
        local_players_.handles.clear();
        for (size_t i = 0; i < sess.num_players(); ++i) local_players_.handles.push_back(i);
        local_inputs_.reset();
        for (auto& f : read_inputs_) f(*this);  // world.run_schedule(ReadInputs)
        if (!local_inputs_)
            throw Panic(BGR_ERR_MISSING_RESOURCE, "No local player inputs found. Did you insert systems into the ReadInputs schedule?");
        for (auto& kv : local_inputs_->inputs) sess.add_local_input(kv.first, kv.second);
        std::vector<ggrs::GgrsRequest> requests;
        ggrs::MismatchedChecksum err;
        if (sess.advance_frame(requests, err)) {
            bgr_session_info info{BGR_SESSION_SYNCTEST, uint32_t(sess.max_prediction()), uint32_t(sess.check_distance()), 0};
            handle_requests(requests, info, [&](ggrs::Frame f, unsigned __int128 c) { sess.save_cell(f, c); });
        } else {  // :104-115
            SyncTestMismatch ev{err.current_frame, err.mismatched_frames};
            for (auto& o : observers_) o(ev);
        }
    }

    // handle_requests (schedule_systems.rs:170-289): ONE C-ABI call for the whole vector
    void handle_requests(const std::vector<ggrs::GgrsRequest>& requests, const bgr_session_info& info,
                         const std::function<void(ggrs::Frame, unsigned __int128)>& save_cell) {
        std::vector<bgr_request> reqs(requests.size());
        for (size_t i = 0; i < requests.size(); ++i) {
            bgr_request& q = reqs[i];
            std::memset(&q, 0, sizeof q);
            q.kind = uint32_t(requests[i].kind);
            q.frame = requests[i].frame;
            q.n_players = uint32_t(requests[i].inputs.size());
            for (size_t p = 0; p < requests[i].inputs.size() && p < BGR_MAX_PLAYERS; ++p) {
                q.inputs[p] = requests[i].inputs[p].first;
                q.status[p] = uint8_t(requests[i].inputs[p].second);
            }
        }
        last_checksums_.assign(BGR_MAX_REQUESTS, bgr_checksum{});
        uint32_t n = 0;
        check(bgr_handle_requests(engine_, &info, reqs.data(), uint32_t(reqs.size()), last_checksums_.data(), BGR_MAX_REQUESTS, &n));
        last_checksums_.resize(n);
        if (!resources_.empty()) handle_resource_requests(requests);
        if (!host_cols_.empty()) handle_host_component_requests(requests);
        for (auto& cs : last_checksums_)  // cell.save(frame, None, checksum) (:231-236)
            save_cell(cs.frame, (static_cast<unsigned __int128>(cs.hi) << 64) | cs.lo);
    }

    // host-side half of handle_requests for resources: the same request vector replayed on a few bytes
    void handle_resource_requests(const std::vector<ggrs::GgrsRequest>& requests) {
        size_t k = 0;
        for (const auto& r : requests) {
            if (r.kind == ggrs::GgrsRequest::SaveGameState) {
                res_store_[res_frame_] = resources_;
                uint64_t part = 0;
                for (auto& t : res_checksummed_) { auto& b = resources_.at(t); part ^= bgr_seahash(b.data(), b.size()); }
                if (k < last_checksums_.size()) last_checksums_[k].lo ^= part;
                ++k;
            } else if (r.kind == ggrs::GgrsRequest::LoadGameState) {
                res_frame_ = r.frame;
                resources_ = res_store_.at(r.frame);
            } else {
                res_frame_ += 1;
                for (auto& f : res_systems_) f(*this);
            }
        }
        int32_t frames[128]; uint32_t nf = 0;
        check(bgr_snapshot_frames(engine_, frames, 128, &nf));
        for (auto it = res_store_.begin(); it != res_store_.end();) {
            bool alive = false;
            for (uint32_t i = 0; i < nf && i < 128; ++i) alive = alive || frames[i] == it->first;
            it = alive ? std::next(it) : res_store_.erase(it);
        }
    }

    // host-side half of handle_requests for non-POD components (see rollback_component_with_clone)
    struct HostColumnBase {
        virtual ~HostColumnBase() = default;
        virtual void save(ggrs::Frame f) = 0;
        virtual void load(ggrs::Frame f) = 0;
        virtual void prune(const std::vector<uint8_t>& alive, const std::vector<int32_t>& kept_frames) = 0;
        virtual bool empty() const = 0;
    };
    template <class T> struct HostColumn : HostColumnBase {
        std::map<uint32_t, T> live;
        std::map<ggrs::Frame, std::map<uint32_t, T>> snaps;
        void save(ggrs::Frame f) override { snaps[f] = live; }  // T's copy constructor is its Clone
        void load(ggrs::Frame f) override {
            auto it = snaps.find(f);
            if (it == snaps.end())  // mod.rs:209-212
                throw Panic(BGR_ERR_NO_SNAPSHOT, "Could not rollback to " + std::to_string(f) + ": no snapshot at that moment could be found.");
            live = it->second;
        }
        void prune(const std::vector<uint8_t>& alive, const std::vector<int32_t>& kept) override {
            for (auto it = live.begin(); it != live.end();)  // the components of despawned entities are gone with them
                it = it->first < alive.size() && alive[it->first] ? std::next(it) : live.erase(it);
            for (auto it = snaps.begin(); it != snaps.end();)  // what the engine's ring discarded (mod.rs:144-199)
                it = std::find(kept.begin(), kept.end(), it->first) != kept.end() ? std::next(it) : snaps.erase(it);
        }
        bool empty() const override { return live.empty(); }
    };
    template <class T> HostColumn<T>& host_col() {
        auto it = host_cols_.find(std::type_index(typeid(T)));
        if (it == host_cols_.end()) throw Panic(BGR_ERR_INVALID_ARGUMENT, std::string("not registered for rollback: ") + typeid(T).name());
        return static_cast<HostColumn<T>&>(*it->second);
    }
    bool entity_exists(uint32_t row) {
        finish();
        uint32_t rows = 0;
        check(bgr_row_count(engine_, &rows));
        if (row >= rows) return false;
        uint8_t a = 0;
        check(bgr_read_alive(engine_, row, 1, &a));
        return a != 0;
    }
    void handle_host_component_requests(const std::vector<ggrs::GgrsRequest>& requests) {
        for (const auto& r : requests) {
            if (r.kind == ggrs::GgrsRequest::SaveGameState) for (auto& c : host_cols_) c.second->save(r.frame);
            else if (r.kind == ggrs::GgrsRequest::LoadGameState) for (auto& c : host_cols_) c.second->load(r.frame);
        }
        std::vector<uint8_t> alive;
        bool any = false;
        for (auto& c : host_cols_) any = any || !c.second->empty();
        if (any) {
            uint32_t rows = 0;
            check(bgr_row_count(engine_, &rows));
            alive.resize(rows);
            if (rows) check(bgr_read_alive(engine_, 0, rows, alive.data()));
        }
        const std::vector<int32_t> kept = snapshot_frames();
        for (auto& c : host_cols_) c.second->prune(alive, kept);
    }
    std::map<std::type_index, std::unique_ptr<HostColumnBase>> host_cols_;

    struct PendingCol { std::type_index type; std::string name; uint32_t bytes, strategy; };
    using ResourceMap = std::map<std::type_index, std::vector<uint8_t>>;
    ResourceMap resources_;
    std::vector<std::type_index> res_checksummed_;
    std::vector<std::function<void(App&)>> res_systems_;
    std::map<ggrs::Frame, ResourceMap> res_store_;
    ggrs::Frame res_frame_ = 0;
    bgr_config cfg_{};
    bgr_engine* engine_ = nullptr;
    std::vector<PendingCol> pending_cols_;
    std::map<std::type_index, uint32_t> columns_;
    std::vector<std::pair<uint32_t, ByteRangeHasher>> checksums_;
    std::vector<System> systems_;
    std::vector<CudaSystem> cuda_systems_;  // parallel to systems_: a non-empty name marks a user system
    std::vector<std::function<void(App&)>> read_inputs_, startup_;
    std::vector<std::function<void(const SyncTestMismatch&)>> observers_;
    std::optional<Session> session_;
    std::optional<LocalInputs> local_inputs_;
    LocalPlayers local_players_;
    std::vector<bgr_checksum> last_checksums_;
    uint64_t accumulator_ns_ = 0;
    bool run_slow_ = false, first_update_ = true;
};

}  // namespace bevy_ggrs
