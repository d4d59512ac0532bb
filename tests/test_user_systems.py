"""User systems (bgr_add_user_system) without a GPU: the generated kernel's prelude with user sources compiles for sm_100a,
the invocation glue stays in registers, compile errors come back with NVRTC's log, and the oracle running CPU builds of
the same sources restates the contract."""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from bevy_ggrs_b200 import capi
from bevy_ggrs_b200.plugin import App, CudaSystem, GgrsPlugin, GgrsSchedule, LocalInputs, ReadInputs, RollbackFrameRate, Session
from bevy_ggrs_b200.session import ADVANCE, SAVE, Request, SyncTestSession
from bevy_ggrs_b200.stress import populate, register_particles, synth_particles
from oracle_backend import OracleWorld
from user_system_util import (DRAG_SRC, PARTICLES_DESPAWN_SRC, PARTICLES_UPDATE_SRC, UserOracleWorld, nvrtc_compile, prelude,
                              register_particles_user)

# particles schema: Transform planes 0..9, Velocity 10..12, Ttl 13..14; checksums Velocity (slot 0), translation (slot 1)
P_HASHES = [(10, 0, 12, 1, 0, 0), (0, 0, 12, 1, 1, 0)]
P_USERS = [("update_particles", PARTICLES_UPDATE_SRC, [("Transform", 40, 0), ("Velocity", 12, 10)], []),
           ("despawn_particles", PARTICLES_DESPAWN_SRC, [("Ttl", 8, 13)], [])]
P_USER_SYSTEMS = [("USER", 0, 0, 0, 0), ("USER", 13, 0, 0, 1)]
P_BUILTIN_SYSTEMS = [("BGR_SYS_PARTICLES_UPDATE", 0, 10, 0, 0), ("BGR_SYS_PARTICLES_DESPAWN", 13, 0, 0, 0)]

# mixed world: Score (u32, optional: absent bit 2), Health (u32, optional: 4), Vel (3 x f32), Tag (u32 x 2)
SCORE_SRC = r"""
struct Score { unsigned int v; };
struct Vel { float x, y, z; };
BGR_SYSTEM_FN void score_from_inputs(const bgr_sys_ctx& ctx, bgr_commands&, Score& s, const Vel& v) {
    const unsigned int handle = unsigned(ctx.order % 8u);
    const unsigned int in = handle < ctx.n_players ? ctx.inputs[handle] : 0u;
    s.v = s.v * 3u + in + unsigned(ctx.frame) + ctx.params[1] + (v.x > 0.0f ? 1u : 0u);
}
"""
MIX_DRAG_SRC = r"""
struct Vel { float x, y, z; };
struct Health { unsigned int hp; };
BGR_SYSTEM_FN void drag_and_wear(const bgr_sys_ctx& ctx, bgr_commands& cmd, Vel& v, Health& h) {
    const float k = bgr_f32(ctx.params[0]);
    v.x = v.x * k + ctx.dt; v.y = v.y * k; v.z = sqrtf(v.z * v.z + 1.0f);
    h.hp = h.hp > 2u ? h.hp - 2u : 0u;
    if (h.hp == 0u) cmd.despawn();
}
"""
M_HASHES = [(0, 0, 4, 0, 0, 2), (1, 0, 4, 0, 1, 4), (2, 0, 12, 1, 2, 0), (5, 0, 8, 0, 3, 0)]
M_USERS = [("score_from_inputs", SCORE_SRC, [("Score", 4, 0), ("Vel", 12, 2)], [0, 7]),
           ("drag_and_wear", MIX_DRAG_SRC, [("Vel", 12, 2), ("Health", 4, 1)], [0x3F733333])]
M_SYSTEMS = [("BGR_SYS_U32_ADD", 0, 0, 2, 1), ("USER", 0, 0, 2, 0), ("USER", 2, 0, 4, 1)]

CONST_SRC = r"""
struct Vel { float x, y, z; };
struct Tag { unsigned int a, b; };
BGR_SYSTEM_FN void tag_from_vel(const bgr_sys_ctx&, bgr_commands&, const Vel& v, Tag& t) {
    t.a = t.a ^ (v.x < 0.0f ? 1u : 2u); t.b = t.b + 1u;
}
"""
C_USERS = [("tag_from_vel", CONST_SRC, [("Vel", 12, 2), ("Tag", 8, 5)], [])]


@pytest.mark.parametrize("rows,item_rows", [(1, 512), (2, 512), (4, 512), (4, 128), (2, 128)])
@pytest.mark.parametrize("world", ["particles", "mixed", "const_binding"])
def test_user_source_prelude_compiles_for_sm_100a(world, rows, item_rows):
    if world == "particles":
        pre = prelude(15, rows, item_rows, P_USER_SYSTEMS, P_HASHES, P_USERS)
    elif world == "mixed":
        pre = prelude(7, rows, item_rows, M_SYSTEMS, M_HASHES, M_USERS)
    else:
        pre = prelude(7, rows, item_rows, [("USER", 2, 0, 0, 0)], M_HASHES, C_USERS)
    rc, log, cubin = nvrtc_compile(pre)
    assert rc == 0, log
    assert cubin[:4] == b"\x7fELF" and b"k_generic_jit" in cubin


def _cuobjdump(cubin, *args):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not installed")
    with tempfile.NamedTemporaryFile(suffix=".cubin", delete=False) as f:
        f.write(cubin)
    try:
        return subprocess.run([exe, *args, f.name], capture_output=True, text=True, check=True).stdout
    finally:
        os.unlink(f.name)


def _resources(cubin):
    import re
    res = _cuobjdump(cubin, "-res-usage")
    line = next(l for l in res.splitlines() if "REG:" in l)
    reg = int(re.search(r"REG:(\d+)", line).group(1))
    stack = int(re.search(r"STACK:(\d+)", line).group(1))
    local = int(re.search(r"LOCAL:(\d+)", line).group(1))
    sass = _cuobjdump(cubin, "-sass")
    n_instr = sum(1 for l in sass.splitlines() if re.match(r"\s+/\*[0-9a-f]{4}\*/\s+\S", l))
    return reg, stack, local, n_instr


@pytest.mark.parametrize("rows,item_rows", [(4, 512), (2, 128)])
def test_user_source_particles_kernel_stays_in_registers(rows, item_rows):
    """The glue (typed locals memcpy'd from literal word planes) disappears after inlining: no stack, no local memory, and
    the same register count and code size as the kernel of the compiled-in update / despawn systems."""
    rc, log, user = nvrtc_compile(prelude(15, rows, item_rows, P_USER_SYSTEMS, P_HASHES, P_USERS))
    assert rc == 0, log
    rc, log, builtin = nvrtc_compile(prelude(15, rows, item_rows, P_BUILTIN_SYSTEMS, P_HASHES))
    assert rc == 0, log
    ru, rb = _resources(user), _resources(builtin)
    assert ru[1] == 0 and ru[2] == 0, f"user-source kernel: STACK:{ru[1]} LOCAL:{ru[2]}"
    assert abs(ru[0] - rb[0]) <= 0.05 * rb[0], f"registers: user {ru[0]}, built-in {rb[0]}"
    assert abs(ru[3] - rb[3]) <= 0.05 * rb[3], f"SASS instructions: user {ru[3]}, built-in {rb[3]}"


def _compile_error(users, systems=None):
    rc, log, _ = nvrtc_compile(prelude(7, 4, 512, systems or [("USER", 2, 0, 0, 0)], M_HASHES, users))
    assert rc != 0
    return log


def test_size_mismatch_names_the_column():
    src = "struct Vel { float x, y; };\nBGR_SYSTEM_FN void f(const bgr_sys_ctx&, bgr_commands&, Vel& v) { v.x = 1.0f; }\n"
    log = _compile_error([("f", src, [("Velocity", 12, 2)], [])])
    assert "column 'Velocity' of 12 bytes" in log, log


def test_write_to_a_const_binding_is_an_error():
    src = "struct Vel { float x, y, z; };\nBGR_SYSTEM_FN void f(const bgr_sys_ctx&, bgr_commands&, const Vel& v) {\n    v.x = 1.0f;\n}\n"
    log = _compile_error([("f", src, [("Vel", 12, 2)], [])])
    assert "f(3)" in log and "error" in log, log


def test_syntax_error_reports_the_users_line():
    src = "struct Vel { float x, y, z; };\n\nBGR_SYSTEM_FN void g(const bgr_sys_ctx&, bgr_commands&, Vel& v) {\n    v.x = v.x * ;\n}\n"
    log = _compile_error([("g", src, [("Vel", 12, 2)], [])])
    assert "g(4)" in log, log


# ---- oracle ----
def _drag_world(n, params, seed=3):
    w = UserOracleWorld(fps=60)
    v = w.rollback_component("Velocity", 12)
    w.checksum_component(v, 0, 12)
    w.add_user_system("apply_drag", DRAG_SRC, [v], params)
    w.build()
    w.spawn(n)
    rng = np.random.default_rng(seed)
    vel = rng.uniform(-2.0, 2.0, (n, 3)).astype(np.float32)
    vel[: n // 4, :2] = 0.0  # these despawn on the first frame
    w.write_component(v, 0, vel)
    return w, v, vel


def test_oracle_user_system_matches_numpy_restatement_through_synctest():
    """apply_drag (v *= k; despawn when x == y == 0) in float32, through a SyncTest run with rollbacks."""
    n, d, k = 64, 3, np.float32(0.75)
    w, v, vel = _drag_world(n, [int(np.array([k]).view(np.uint32)[0])])
    sess = SyncTestSession(1, d, 8, input_delay=0)
    frames = 12
    for _ in range(frames):
        reqs = sess_requests(sess)
        w.handle_requests(sess.info(), reqs)
    # every frame ran exactly once more than it was rolled back: the live state is `frames` applications
    expect = vel.copy()
    alive = np.ones(n, bool)
    for _ in range(frames):
        expect = (expect * k).astype(np.float32)
        alive &= ~((expect[:, 0] == 0.0) & (expect[:, 1] == 0.0))
    got, has = w.read_component_alive(v, 0, n)
    assert np.array_equal(has.astype(bool), alive)
    assert np.array_equal(got[alive].view(np.float32).reshape(-1, 3), expect[alive])
    w.close()


def sess_requests(sess):
    for h in range(sess.num_players()):
        sess.add_local_input(h, 0)
    return sess.advance_frame()


def _particles_checksums(world_factory, register, n=700, ticks=10):
    w = world_factory()
    cols = register(w)
    w.build()
    tf, vel, ttl = synth_particles(n, 9, 3, 12)
    populate(w, cols, tf, vel, ttl)
    sess = SyncTestSession(2, 4, 8, input_delay=2)
    out = []
    for _ in range(ticks):
        out += w.handle_requests(sess.info(), sess_requests(sess))
    state = [w.read_component_alive(c, 0, n) for c in cols]
    w.close()
    return out, state


def test_oracle_user_particles_give_the_builtin_checksums():
    a, sa = _particles_checksums(lambda: OracleWorld(fps=60), register_particles)
    b, sb = _particles_checksums(lambda: UserOracleWorld(fps=60), register_particles_user)
    assert a == b and len(a) > 10
    for (va, ha), (vb, hb) in zip(sa, sb):
        assert np.array_equal(ha, hb) and np.array_equal(va[ha.astype(bool)], vb[hb.astype(bool)])
    assert 0 < sa[2][1].sum() < 700  # some particles ran out of Ttl inside the run


def test_app_mirror_accepts_cuda_systems():
    """plugin.App hands a CudaSystem to the backend's add_user_system, in add_systems order."""
    w = UserOracleWorld(fps=60)
    app = App(w).add_plugins(GgrsPlugin()).insert_resource(RollbackFrameRate(60))
    app.add_systems(ReadInputs, lambda a: a.insert_resource(LocalInputs({h: 0 for h in a.local_players.handles})))
    v = app.rollback_component_with_copy("Velocity", 12)
    app.checksum_component(v, 0, 12)
    app.add_systems(GgrsSchedule, CudaSystem("apply_drag", DRAG_SRC, [v], [0x3F000000]))
    assert w._systems[0][0] == "user"
    app.insert_resource(Session.SyncTest(SyncTestSession(1, 2, 8, input_delay=0)))
    app._finish()
    w.spawn(4)
    w.write_component(v, 0, np.full((4, 3), 2.0, np.float32))
    for _ in range(3):
        app.step()
    got = w.read_component(v, 0, 4).view(np.float32)
    assert np.all(got == np.float32(0.25))
    w.close()
