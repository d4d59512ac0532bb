"""Test helpers for user systems (bgr_add_user_system): the generated kernel's prelude written out here, NVRTC without a
GPU, and the oracle running a CPU build of the same source.

TEST INFRASTRUCTURE: nothing in the product package imports this file.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
from typing import List, Sequence, Tuple

from bevy_ggrs_b200 import capi
from oracle_backend import OracleWorld

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "bevy_ggrs_b200", "csrc")
TESTS = os.path.dirname(os.path.abspath(__file__))
# jit.hpp's source list
FILES = ["generic_program_jit.cuh", "generic_program.cuh", "kernels.cuh", "seahash.cuh", "tma_copy.cuh", "rtc_prelude.cuh",
         "user_system.cuh"]
SYS_USER = 0x100  # engine.cu kSysUser

# ---- the particles stress systems written as user source (particles.rs:272-289) ----
PARTICLES_UPDATE_SRC = r"""
struct Transform { float translation[3]; float rotation[4]; float scale[3]; };
struct Velocity { float x, y, z; };
BGR_SYSTEM_FN void update_particles(const bgr_sys_ctx& ctx, bgr_commands&, Transform& t, Velocity& v) {
    const float gx = 0.0f * 200.0f, gy = -1.0f * 200.0f, gz = 0.0f * 200.0f;  // Vec3::NEG_Y * 200.0
    v.x = v.x + gx * ctx.dt; v.y = v.y + gy * ctx.dt; v.z = v.z + gz * ctx.dt;
    t.translation[0] = t.translation[0] + v.x * ctx.dt;
    t.translation[1] = t.translation[1] + v.y * ctx.dt;
    t.translation[2] = t.translation[2] + v.z * ctx.dt;
}
"""
PARTICLES_DESPAWN_SRC = r"""
struct Ttl { unsigned long long frames; };
BGR_SYSTEM_FN void despawn_particles(const bgr_sys_ctx&, bgr_commands& cmd, Ttl& ttl) {
    ttl.frames -= 1;
    if (ttl.frames == 0) cmd.despawn();
}
"""
DRAG_SRC = r"""
struct Velocity { float x, y, z; };
BGR_SYSTEM_FN void apply_drag(const bgr_sys_ctx& ctx, bgr_commands& cmd, Velocity& v) {
    const float k = bgr_f32(ctx.params[0]);
    v.x = v.x * k; v.y = v.y * k; v.z = v.z * k;
    if (v.x == 0.0f && v.y == 0.0f) cmd.despawn();
}
"""


def system_ids():
    import re
    hdr = open(os.path.join(ROOT, "include", "bevy_ggrs_b200.h")).read()
    return {m.group(1): int(m.group(2)) for m in re.finditer(r"(BGR_SYS_[A-Z0-9_]+)\s*=\s*(\d+)", hdr)}


def _c_string_literal(text):
    out = '"'
    for ch in text:
        if ch in '"\\':
            out += "\\"
        out += ch if 0x20 <= ord(ch) < 0x7F else "?"
    return out + '"'


def prelude(words, rows, item_rows, systems, hashes, users=()):
    """What engine.cu jit_specialise generates.  systems: (id name | "USER", plane0, plane1, need, param);
    hashes: (first_plane, off, len, finite, slot, absent); users: (name, source, [(column name, elem_bytes, first_plane)],
    params) in registration order."""
    ids = system_ids()
    ids_all = dict(ids, USER=SYS_USER)
    lines = [f"#define {k} {v}" for k, v in ids.items()]
    lines += ["#define BGR_TILE_ROWS 512", f"#define BGR_JIT_WORDS {words}", f"#define BGR_JIT_ROWS {rows}",
              f"#define BGR_JIT_ITEM_ROWS {item_rows}", f"#define BGR_JIT_MINB {max(1, (512 if words <= 8 else 256) // (item_rows // rows))}",
              f"#define BGR_JIT_NSYS {len(systems)}", f"#define BGR_JIT_NHASH {len(hashes)}"]
    fmt = lambda t: "{" + ",".join(f"{int(v)}u" for v in t) + "}"
    lines.append("#define BGR_JIT_SYS_LIST " + ", ".join([fmt((ids_all[s[0]],) + tuple(s[1:])) for s in systems] + ["{0u,0u,0u,0u,0u}"]))
    lines.append("#define BGR_JIT_HASH_LIST " + ", ".join([fmt(h) for h in hashes] + ["{0u,0u,0u,0u,0u,0u}"]))
    pre = "\n".join(lines) + "\n"
    if not users:
        return pre
    pre += f"#define BGR_SYS_USER {SYS_USER}\n#include \"user_system.cuh\"\n"
    for i, (name, source, cols, params) in enumerate(users):
        fn = f"bgr_user_{i}::{name}"
        pre += f"namespace bgr_user_{i} {{\n#line 1 \"{name}\"\n{source}\n}}\n"
        pre += f"#line 1 \"bgr_user_dispatch_{name}\"\n"
        pre += f"template <> struct bgr_user_system<{i}> {{\n"
        pre += f"    using F = bgr_fn_traits<decltype(&{fn})>;\n"
        pre += (f"    static_assert(F::arity == {len(cols)}, "
                + _c_string_literal(f"{name}: takes one component parameter per bound column ({len(cols)})") + ");\n")
        for j, (cname, eb, _plane) in enumerate(cols):
            msg = f"{name}: parameter {j + 1} is bound to column '{cname}' of {eb} bytes; sizeof of the parameter type differs"
            pre += f"    static_assert(sizeof(F::elem<{j}>) == {eb}, " + _c_string_literal(msg) + ");\n"
        pre += "    template <int N> static __device__ __forceinline__ void run(uint32_t (&w)[N], bool on, const bgr_sys_ctx& base, bool& kill) {\n"
        pre += "        bgr_sys_ctx ctx = base;\n"
        for j in range(8):
            pre += f"        ctx.params[{j}] = {params[j] if j < len(params) else 0}u;\n"
        planes = ", ".join(str(c[2]) for c in cols)
        pre += f"        bgr_invoke<&{fn}>::run<{planes}>(w, on, ctx, kill);\n    }}\n}};\n"
    return pre


def nvrtc():
    import pytest
    for name in ("libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so"):
        try:
            return C.CDLL(name)
        except OSError:
            continue
    pytest.skip("libnvrtc not installed")


def nvrtc_compile(pre) -> Tuple[int, str, bytes]:
    """(status, log, cubin) of prelude + generic_program_jit.cuh, with the engine's options."""
    lib = nvrtc()
    contents = [open(os.path.join(CSRC, f), "rb").read() for f in FILES]
    prog = C.c_void_p()
    hs = (C.c_char_p * len(FILES))(*contents)
    ns = (C.c_char_p * len(FILES))(*[f.encode() for f in FILES])
    src = (pre + '#include "generic_program_jit.cuh"\n').encode()
    assert lib.nvrtcCreateProgram(C.byref(prog), src, b"bgr_generic_jit.cu", len(FILES), hs, ns) == 0
    opts = [b"--gpu-architecture=sm_100a", b"-std=c++17", b"-fmad=false", b"-lineinfo"]
    rc = lib.nvrtcCompileProgram(prog, len(opts), (C.c_char_p * len(opts))(*opts))
    n = C.c_size_t()
    lib.nvrtcGetProgramLogSize(prog, C.byref(n))
    log = C.create_string_buffer(n.value)
    lib.nvrtcGetProgramLog(prog, log)
    cubin = b""
    if rc == 0:
        lib.nvrtcGetCUBINSize(prog, C.byref(n))
        buf = C.create_string_buffer(n.value)
        lib.nvrtcGetCUBIN(prog, buf)
        cubin = buf.raw
    lib.nvrtcDestroyProgram(C.byref(prog))
    return rc, log.value.decode(errors="replace"), cubin


# ---- the oracle running CPU builds of user sources ----
def build_host_library(sources: Sequence[Tuple[str, str]]) -> str:
    """One shared library: the oracle's user-system extension (user_system_oracle.cpp) + every (name, source), each in its
    own namespace, with a C trampoline `usr_tramp_<i>`.  Built in a temporary directory, cached by content."""
    text = f'#include "{os.path.join(TESTS, "user_system_oracle.cpp")}"\n'
    for i, (name, src) in enumerate(sources):
        text += f"namespace usr_{i} {{\n#line 1 \"{name}\"\n{src}\n}}\n"
        text += (f'extern "C" __attribute__((visibility("default"))) void usr_tramp_{i}(const bgr_sys_ctx* c, uint8_t* const* e, int* d) '
                 f"{{ usr_call(&usr_{i}::{name}, c, e, d); }}\n")
    deps = "".join(open(os.path.join(p), encoding="utf-8").read() for p in (
        os.path.join(TESTS, "user_system_oracle.cpp"), os.path.join(CSRC, "user_system.cuh"), os.path.join(ROOT, "oracle", "world.hpp")))
    key = hashlib.sha256((text + deps).encode()).hexdigest()[:20]
    out_dir = os.path.join(tempfile.gettempdir(), f"bgr_user_host_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.join(out_dir, f"libusr_{key}.so")
    if not os.path.exists(out):
        cpp = os.path.join(out_dir, f"usr_{key}.cpp")
        with open(cpp, "w") as f:
            f.write(text)
        tmp = out + f".{os.getpid()}.tmp"
        cmd = ["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-fvisibility=hidden",
               "-pthread", "-o", tmp, cpp]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("host build of user systems failed:\n" + r.stderr)
        os.replace(tmp, out)
    return out


class UserOracleWorld(OracleWorld):
    """OracleWorld that also runs user systems, from a CPU build of their source.  Systems are registered at build() in
    add_systems order (the library holding the user sources is compiled then)."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self._systems: List[tuple] = []
        self._usr = None

    def add_system(self, system, cols, params=()):
        self._systems.append(("builtin", system, list(cols), list(params)))

    def add_user_system(self, name, source, cols, params=()):
        self._systems.append(("user", (name, source), list(cols), list(params)))

    def build(self):
        users = [s[1] for s in self._systems if s[0] == "user"]
        if users:
            self._usr = C.CDLL(build_host_library(users))
            u32, vp = C.c_uint32, C.c_void_p
            self._usr.usr_add_user_system.argtypes = [vp, vp, C.POINTER(u32), u32, C.POINTER(u32), u32]
            self._usr.usr_handle_requests.argtypes = [vp, C.POINTER(capi.bgr_session_info), C.POINTER(capi.bgr_request), u32,
                                                      C.POINTER(capi.bgr_checksum), u32, C.POINTER(u32)]
            self._usr.usr_advance_world.argtypes = [vp, vp, u32]
            self._usr.usr_forget_world.argtypes = [vp]
            self._usr.usr_last_error.restype = C.c_char_p
        k = 0
        for kind, what, cols, params in self._systems:
            if kind == "builtin":
                super().add_system(what, cols, params)
                continue
            ca = (C.c_uint32 * max(1, len(cols)))(*cols)
            pa = (C.c_uint32 * max(1, len(params)))(*params)
            fn = C.cast(getattr(self._usr, f"usr_tramp_{k}"), C.c_void_p)
            self._check_usr(self._usr.usr_add_user_system(self._h, fn, ca, len(cols), pa, len(params)))
            k += 1

    def _check_usr(self, st):
        if st != 0:
            from oracle_backend import OracleError
            raise OracleError(st, self._usr.usr_last_error().decode())

    def advance_world(self, inputs=(), status=()):
        if self._usr is None:
            return super().advance_world(inputs, status)
        ia = (C.c_uint8 * capi.BGR_MAX_PLAYERS)(*[v & 0xFF for v in inputs])
        self._check_usr(self._usr.usr_advance_world(self._h, ia, len(inputs)))

    def handle_requests(self, session_info, requests):
        if self._usr is None:
            return super().handle_requests(session_info, requests)
        reqs = list(requests)
        arr = capi.make_requests(reqs)
        info = capi.make_session_info(session_info)
        out = (capi.bgr_checksum * capi.BGR_MAX_REQUESTS)()
        n = C.c_uint32()
        st = self._usr.usr_handle_requests(self._h, C.byref(info), arr, len(reqs), out, capi.BGR_MAX_REQUESTS, C.byref(n))
        self._check_usr(st)
        return [(out[i].frame, (out[i].hi << 64) | out[i].lo) for i in range(n.value)]

    def close(self):
        if self._usr is not None and self._h:
            self._usr.usr_forget_world(self._h)
        super().close()


def register_particles_user(world):
    """stress.register_particles with update_particles / despawn_particles given as user source."""
    t = world.rollback_component("Transform", 40, capi.BGR_STRATEGY_CLONE)
    v = world.rollback_component("Velocity", 12, capi.BGR_STRATEGY_COPY)
    l = world.rollback_component("Ttl", 8, capi.BGR_STRATEGY_COPY)
    world.checksum_component(v, 0, 12, capi.BGR_HASH_FLAG_ASSERT_FINITE_F32)
    world.checksum_component(t, 0, 12, capi.BGR_HASH_FLAG_ASSERT_FINITE_F32)
    world.add_user_system("update_particles", PARTICLES_UPDATE_SRC, [t, v])
    world.add_user_system("despawn_particles", PARTICLES_DESPAWN_SRC, [l])
    return t, v, l
