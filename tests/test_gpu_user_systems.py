"""User systems (bgr_add_user_system) on the GPU: CUDA source compiled into the registration's own kernel at bgr_build,
checked bit for bit against the oracle.  Every case runs on whole-tile and quarter-tile work items (the two instances of
the generated kernel) at 3 000 and 120 000 entities.  User systems have no interpreter arm, so this module declares its own
fixture instead of conftest's `generic_kernel`."""

import numpy as np
import pytest

from bevy_ggrs_b200 import capi
from bevy_ggrs_b200.capi import BgrError
from bevy_ggrs_b200.engine import Engine
from bevy_ggrs_b200.plugin import (App, CudaSystem, GgrsPlugin, GgrsSchedule, LocalInputs, ReadInputs, RollbackFrameRate,
                                   Session, SyncTestMismatch)
from bevy_ggrs_b200.session import ADVANCE, LOAD, SAVE, P2PTraceSession, Request, SyncTestSession
from bevy_ggrs_b200.stress import populate, register_particles, synth_particles
from oracle_backend import OracleWorld
from user_system_util import (DRAG_SRC, UserOracleWorld,
                              register_particles_user)

pytestmark = pytest.mark.gpu
SIZES = [3000, 120000]

SCORE_SRC = r"""
struct Score { unsigned int v; };
struct Vel { float x, y, z; };
BGR_SYSTEM_FN void score_from_inputs(const bgr_sys_ctx& ctx, bgr_commands&, Score& s, const Vel& v) {
    const unsigned int handle = unsigned(ctx.order % 8u);
    const unsigned int in = handle < ctx.n_players ? ctx.inputs[handle] : 0u;
    s.v = s.v * 3u + in + unsigned(ctx.frame) + ctx.params[1] + (v.x > 0.0f ? 1u : 0u);
}
"""
WEAR_SRC = r"""
struct Vel { float x, y, z; };
struct Health { unsigned int hp; };
BGR_SYSTEM_FN void drag_and_wear(const bgr_sys_ctx& ctx, bgr_commands& cmd, Vel& v, Health& h) {
    const float k = bgr_f32(ctx.params[0]);
    v.x = v.x * k + ctx.dt; v.y = v.y * k; v.z = sqrtf(v.z * v.z + 1.0f);
    h.hp = h.hp > 2u ? h.hp - 2u : 0u;
    if (h.hp == 0u) cmd.despawn();
}
"""
TIMER_SRC = r"""
struct Score { unsigned int v; };
BGR_SYSTEM_FN void stamp_time(const bgr_sys_ctx&, bgr_commands&, Score& s) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    s.v = unsigned(t);
}
"""


@pytest.fixture(params=["whole_tiles", "quarter_tiles"])
def item(request, monkeypatch):
    """The generated kernel with one tile (512 rows) or a quarter tile (128 rows) per work item."""
    monkeypatch.setenv("BGR_TUNE_JIT_ITEM", "512" if request.param == "whole_tiles" else "128")
    return request.param


def _drive(worlds, sessions, ticks):
    """Same request vectors to every world; returns each world's checksums."""
    out = [[] for _ in worlds]
    for _ in range(ticks):
        reqs = []
        for s in sessions:
            for h in range(s.num_players()):
                s.add_local_input(h, 0)
            reqs.append(s.advance_frame())
        for i, (w, s, r) in enumerate(zip(worlds, sessions, reqs)):
            cs = w.handle_requests(s.info(), r)
            for f, c in cs:
                s.save_cell(f, c)
            out[i] += cs
    return out


def _same_state(eng, orc, cols, n):
    alive = eng.read_alive(0, n).astype(bool)
    assert np.array_equal(alive, orc.read_alive(0, n).astype(bool)), "alive mask"
    for c in cols:
        vo, ho = orc.read_component_alive(c, 0, n)
        he = ho.astype(bool)
        assert np.array_equal(eng.read_component(c, 0, n)[he], vo[he]), f"column {c}"


def _particles_pair(n, depth):
    eng = Engine(max_entities=n, max_depth=depth)
    orc = OracleWorld(fps=60)
    cols = register_particles_user(eng)
    register_particles(orc)   # the oracle's compiled-in systems: it does not share the user source
    eng.build()
    orc.build()
    assert eng.generic_specialised()
    data = synth_particles(n, 21, 3, 40, z_fraction=0.1)
    populate(eng, cols, *data)
    populate(orc, cols, *data)
    return eng, orc, cols


@pytest.mark.parametrize("n", SIZES)
def test_user_particles_match_builtin_oracle_synctest_and_p2p(item, n):
    d = 8
    eng, orc, cols = _particles_pair(n, d + 1)
    a, b = _drive([eng, orc], [SyncTestSession(2, d, d + 1, input_delay=2), SyncTestSession(2, d, d + 1, input_delay=2)], 14)
    assert a == b and len(a) > 20
    assert eng.last_path_fused()
    _same_state(eng, orc, cols, n)
    eng.close(); orc.close()
    eng, orc, cols = _particles_pair(n, 9)
    a, b = _drive([eng, orc], [P2PTraceSession(2, 8, 2, seed=5), P2PTraceSession(2, 8, 2, seed=5)], 24)
    assert a == b and len(a) >= 24
    _same_state(eng, orc, cols, n)
    assert 0 < orc.active_count() < n  # Ttl ran out for some particles
    eng.close(); orc.close()


def _mixed_pair(n, depth, flags=0, order_base=0, first=0, count=None):
    """Built-in U32_ADD on Score + two user systems on optional columns; the oracle runs CPU builds of the same source."""
    count = n if count is None else count
    worlds = []
    for w in (Engine(max_entities=count, max_depth=depth, flags=flags, order_base=order_base),
              UserOracleWorld(fps=60, order_base=order_base)):
        score = w.rollback_component("Score", 4, capi.BGR_STRATEGY_COPY | capi.BGR_STRATEGY_OPTIONAL)
        health = w.rollback_component("Health", 4, capi.BGR_STRATEGY_CLONE | capi.BGR_STRATEGY_OPTIONAL)
        vel = w.rollback_component("Vel", 12, capi.BGR_STRATEGY_COPY)
        tag = w.rollback_component("Tag", 8, capi.BGR_STRATEGY_COPY)
        w.checksum_component(score, 0, 4)
        w.checksum_component(health, 0, 4)
        w.checksum_component(vel, 0, 12, capi.BGR_HASH_FLAG_ASSERT_FINITE_F32)
        w.checksum_component(tag, 0, 8)
        w.add_system(capi.BGR_SYS_U32_ADD, [score], [0, 1])
        w.add_user_system("score_from_inputs", SCORE_SRC, [score, vel], [0, 7])
        w.add_user_system("drag_and_wear", WEAR_SRC, [vel, health], [0x3F733333])
        w.build()
        w.spawn(count)
        rng = np.random.default_rng(17)
        w.write_component(score, 0, rng.integers(0, 1000, n, dtype=np.uint32)[first:first + count])
        w.write_component(health, 0, rng.integers(4, 60, n, dtype=np.uint32)[first:first + count])
        w.write_component(vel, 0, rng.uniform(-3, 3, (n, 3)).astype(np.float32)[first:first + count])
        w.write_component(tag, 0, rng.integers(0, 2**32, (n, 2), dtype=np.uint32)[first:first + count])
        worlds.append(w)
    return worlds[0], worlds[1], (score, health, vel, tag)


def _mixed_requests(frame, d, rng):
    """SyncTest-shaped vector with varying inputs for 3 players."""
    inp = lambda: [int(x) for x in rng.integers(0, 256, 3)]
    reqs = []
    if frame >= d:
        reqs.append(Request(LOAD, frame - d))
        for k in range(d):
            reqs.append(Request(ADVANCE, 0, inp()))
            if k < d - 1:
                reqs.append(Request(SAVE, frame - d + k + 1))
    return reqs + [Request(SAVE, frame), Request(ADVANCE, 0, inp())]


@pytest.mark.parametrize("n", SIZES)
def test_mixed_world_matches_oracle_with_presence_changes(item, n):
    d = 4
    eng, orc, cols = _mixed_pair(n, 8)
    score, health = cols[0], cols[1]
    sess = (capi.BGR_SESSION_SYNCTEST, 8, d, 0)
    rng_e, rng_o, rng = np.random.default_rng(2), np.random.default_rng(2), np.random.default_rng(3)
    for frame in range(12):
        l0 = eng.launch_count()
        a = eng.handle_requests(sess, _mixed_requests(frame, d, rng_e))
        b = orc.handle_requests(sess, _mixed_requests(frame, d, rng_o))
        assert a == b, f"frame {frame}"
        assert eng.launch_count() - l0 == 1   # one launch per request vector
        alive = np.flatnonzero(orc.read_alive(0, n))
        for r in rng.choice(alive, min(40, alive.size), replace=False):   # remove / insert between request vectors
            c = (score, health)[int(rng.integers(2))]
            had = bool(orc.has_component(c, int(r), 1)[0])
            value = np.uint32(rng.integers(5, 50))
            for w in (eng, orc):
                if had:
                    w.remove_component(c, int(r))
                else:
                    w.insert_component(c, int(r), value)
        _same_state(eng, orc, cols, n)
    assert 0 < orc.active_count() < n  # drag_and_wear despawned some entities
    eng.close(); orc.close()


def test_specialised_even_for_tiny_worlds(item):
    eng, orc, cols = _mixed_pair(64, 4)
    assert eng.generic_specialised()
    l0 = eng.launch_count()
    a = eng.handle_requests((capi.BGR_SESSION_NONE, 0, 0, 0), [Request(SAVE, 0), Request(ADVANCE, 0, [1, 2]), Request(SAVE, 1)])
    assert eng.launch_count() - l0 == 1
    assert a == orc.handle_requests((capi.BGR_SESSION_NONE, 0, 0, 0), [Request(SAVE, 0), Request(ADVANCE, 0, [1, 2]), Request(SAVE, 1)])
    eng.close(); orc.close()


@pytest.mark.parametrize("n", SIZES)
def test_pipelined_with_tile_dependencies_then_synchronous(item, monkeypatch, n):
    monkeypatch.setenv("BGR_TUNE_JIT_TILEDEP", "1")
    d = 4
    eng, orc, cols = _mixed_pair(n, 8)
    sess = (capi.BGR_SESSION_SYNCTEST, 8, d, 0)
    rng_e, rng_o = np.random.default_rng(4), np.random.default_rng(4)
    got, want = [], []
    for frame in range(12):
        eng.submit_requests(sess, _mixed_requests(frame, d, rng_e))
        want += orc.handle_requests(sess, _mixed_requests(frame, d, rng_o))
        if frame % 4 == 3:   # four vectors in flight
            for _ in range(4):
                got += eng.collect()
    for frame in range(12, 16):
        got += eng.handle_requests(sess, _mixed_requests(frame, d, rng_e))
        want += orc.handle_requests(sess, _mixed_requests(frame, d, rng_o))
    assert got == want
    _same_state(eng, orc, cols, n)
    eng.close(); orc.close()


@pytest.mark.parametrize("n", SIZES)
def test_sharded_pair_equals_unsharded(item, n):
    d = 4
    sess = (capi.BGR_SESSION_SYNCTEST, 8, d, 0)
    half = n // 2 + 7
    whole, _, _ = _mixed_pair(n, 8)
    shards = [_mixed_pair(n, 8, flags=capi.BGR_CFG_SHARDED, order_base=first, first=first, count=count)[0]
              for first, count in ((0, half), (half, n - half))]
    lib = capi.load_library()
    rng = np.random.default_rng(9)
    for frame in range(10):
        reqs = _mixed_requests(frame, d, rng)
        want = whole.handle_requests(sess, reqs)
        parts = []
        for e in shards:
            e.handle_requests(sess, reqs)
            parts.append(e.last_partials())
        comb = (capi.bgr_partial * len(want))()
        for i in range(len(want)):
            comb[i].frame, comb[i].n_columns = parts[0][i].frame, parts[0][i].n_columns
            comb[i].active = sum(p[i].active for p in parts)
            comb[i].total = sum(p[i].total for p in parts)
            for c in range(capi.BGR_MAX_CHECKSUM_COLUMNS):
                comb[i].xor_[c] = parts[0][i].xor_[c] ^ parts[1][i].xor_[c]
        out = (capi.bgr_checksum * len(want))()
        assert lib.bgr_fold_partials_n(comb, len(want), out) == 0
        assert [(o.frame, (o.hi << 64) | o.lo) for o in out] == want, f"frame {frame}"
    for e in [whole] + shards:
        e.close()


def _app(source, name, ticks, n=3000):
    eng = Engine(max_entities=n, max_depth=9)
    app = App(eng).add_plugins(GgrsPlugin()).insert_resource(RollbackFrameRate(60))
    app.add_systems(ReadInputs, lambda a: a.insert_resource(LocalInputs({h: a.ticks % 7 for h in a.local_players.handles})))
    score = app.rollback_component_with_copy("Score", 4)
    vel = app.rollback_component_with_copy("Vel", 12)
    app.checksum_component(score, 0, 4).checksum_component(vel, 0, 12, assert_finite=True)
    app.add_systems(GgrsSchedule, CudaSystem(name, source, [score] if name == "stamp_time" else [score, vel], [0, 3]))
    app.insert_resource(Session.SyncTest(SyncTestSession(2, 4, 8, input_delay=2)))
    mism = []
    app.add_observer(SyncTestMismatch, mism.append)
    app._finish()
    eng.spawn(n)
    eng.write_component(vel, 0, np.random.default_rng(1).uniform(-1, 1, (n, 3)).astype(np.float32))
    for _ in range(ticks):
        app.step()
    eng.close()
    return mism


def test_app_mirror_runs_200_synctest_ticks_without_mismatch(item):
    assert _app(SCORE_SRC, "score_from_inputs", 200) == []


def test_nondeterministic_user_system_fires_synctest_mismatch(item):
    """synctest.rs:83-125: a system that writes what a rollback does not restore into a checksummed column."""
    assert len(_app(TIMER_SRC, "stamp_time", 12)) > 0


def _refused(monkeypatch, env=None, flags=0, source=DRAG_SRC, wide=False, spawn=False, params=(0x3F000000,)):
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    eng = Engine(max_entities=1000, max_depth=4, flags=flags)
    v = eng.rollback_component("Velocity", 12)
    if wide:
        eng.rollback_component("Wide", 88)
    if spawn:
        t = eng.rollback_component("Transform", 40)
        l = eng.rollback_component("Ttl", 8)
        eng.add_system(capi.BGR_SYS_PARTICLES_SPAWN, [t, v, l], [4, 300, 1, 0])
    eng.add_user_system("apply_drag", source, [v], list(params))
    with pytest.raises(BgrError) as ei:
        eng.build()
    eng.close()   # destroyable after the failure
    return ei.value.status, str(ei.value)


def test_refusals(monkeypatch):
    st, text = _refused(monkeypatch, source="struct Velocity { float x, y, z; };\nBGR_SYSTEM_FN void apply_drag(const bgr_sys_ctx&, bgr_commands&, Velocity& v) { v.x = ; }\n")
    assert st == capi.BGR_ERR_INVALID_ARGUMENT and "apply_drag(2)" in text
    assert _refused(monkeypatch, flags=capi.BGR_CFG_FORCE_STEPWISE)[0] == capi.BGR_ERR_UNSUPPORTED
    assert _refused(monkeypatch, wide=True)[0] == capi.BGR_ERR_UNSUPPORTED
    assert _refused(monkeypatch, spawn=True)[0] == capi.BGR_ERR_UNSUPPORTED
    assert _refused(monkeypatch, env={"BGR_TUNE_GENERIC": "0"})[0] == capi.BGR_ERR_UNSUPPORTED
    monkeypatch.delenv("BGR_TUNE_GENERIC")
    assert _refused(monkeypatch, env={"BGR_TUNE_JIT": "0"})[0] == capi.BGR_ERR_UNSUPPORTED
    monkeypatch.delenv("BGR_TUNE_JIT")
    st, text = _refused(monkeypatch, env={"BGR_JIT_SRC_DIR": "/nonexistent"}, params=(0x3F000001,))  # a prelude not compiled before
    assert st == capi.BGR_ERR_UNSUPPORTED and "kernel source not found" in text
    monkeypatch.delenv("BGR_JIT_SRC_DIR")
    # call-time validation
    eng = Engine(max_entities=100, max_depth=4)
    v = eng.rollback_component("Velocity", 12)
    for args, status in ((("2bad", DRAG_SRC, [v]), capi.BGR_ERR_INVALID_ARGUMENT),
                         (("apply_drag", DRAG_SRC, [v, v]), capi.BGR_ERR_INVALID_ARGUMENT),
                         (("apply_drag", DRAG_SRC, [7]), capi.BGR_ERR_INVALID_ARGUMENT),
                         (("apply_drag", "x" * 70000, [v]), capi.BGR_ERR_INVALID_ARGUMENT),
                         (("apply_drag", DRAG_SRC, [v], list(range(9))), capi.BGR_ERR_INVALID_ARGUMENT)):
        with pytest.raises(BgrError) as ei:
            eng.add_user_system(*args)
        assert ei.value.status == status
    eng.add_user_system("apply_drag", DRAG_SRC, [v])
    with pytest.raises(BgrError) as ei:
        eng.add_user_system("apply_drag", DRAG_SRC, [v])
    assert "added twice" in str(ei.value)
    eng.build()
    with pytest.raises(BgrError) as ei:
        eng.add_user_system("later", DRAG_SRC, [v])
    assert ei.value.status == capi.BGR_ERR_STATE
    eng.close()
