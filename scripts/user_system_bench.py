#!/usr/bin/env python
"""Tick time of the particles stress world with update_particles / despawn_particles written as USER SOURCE
(bgr_add_user_system, tests/user_system_util.py) next to the same world on the compiled-in system ids.  Both run with
BGR_TUNE_BUNDLE=0, so both run on the registration's own generated kernel: the difference is the user-system glue alone.
SyncTest d=8 request vectors at 100k and 1M entities, synchronous (handle_requests) and pipelined (4 submits in flight),
the two arms alternated inside one process.  Also records bgr_build's wall time with user sources (NVRTC compile of both
kernel instances).   usage: user_system_bench.py [--ticks K] [--reps R] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

os.environ["BGR_TUNE_BUNDLE"] = "0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from bevy_ggrs_b200.engine import Engine  # noqa: E402
from bevy_ggrs_b200.session import SAVE, SyncTestSession  # noqa: E402
from bevy_ggrs_b200.stress import populate, register_particles, synth_particles  # noqa: E402
from user_system_util import register_particles_user  # noqa: E402

D = 8


def make(n, user):
    eng = Engine(max_entities=n, max_depth=D + 1)
    cols = register_particles_user(eng) if user else register_particles(eng)
    t0 = time.perf_counter()
    eng.build()
    build_s = time.perf_counter() - t0
    assert eng.generic_specialised(), "the generated kernel was not compiled"
    populate(eng, cols, *synth_particles(n, 7, 1_000_000, 1_000_001))  # nobody dies inside the run
    return eng, build_s


def vectors(count):
    s = SyncTestSession(2, D, D + 1, input_delay=2)
    out = []
    for _ in range(count):
        for h in range(2):
            s.add_local_input(h, 0)
        reqs = s.advance_frame()
        for r in reqs:
            if r.kind == SAVE:
                s.save_cell(r.frame, 0)
        out.append(reqs)
    return out, s.info()


def run_block(eng, vecs, info, pipelined):
    t0 = time.perf_counter()
    if pipelined:
        inflight = 0
        for v in vecs:
            eng.submit_requests(info, v)
            inflight += 1
            if inflight == 4:
                eng.collect()
                inflight -= 1
        while inflight:
            eng.collect()
            inflight -= 1
    else:
        for v in vecs:
            eng.handle_requests(info, v)
    return (time.perf_counter() - t0) / len(vecs)


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        return r.stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rows = [{"gpu": gpu_info(), "session": f"SyncTest d={D}", "ticks": a.ticks, "reps": a.reps, "BGR_TUNE_BUNDLE": 0}]
    for n in (100_000, 1_000_000):
        engines = {}
        for arm in ("builtin", "user"):
            eng, build_s = make(n, arm == "user")
            vecs, info = vectors(a.warmup + 2 * a.reps * a.ticks)
            engines[arm] = [eng, vecs, info, 0, build_s]
        res = {arm: {"sync": [], "pipelined": []} for arm in engines}
        for arm, e in engines.items():  # warm up both
            run_block(e[0], e[1][: a.warmup], e[2], False)
            e[3] = a.warmup
        for rep in range(a.reps):
            for mode in ("sync", "pipelined"):
                for arm in (("builtin", "user") if rep % 2 == 0 else ("user", "builtin")):
                    e = engines[arm]
                    block = e[1][e[3]: e[3] + a.ticks]
                    e[3] += a.ticks
                    res[arm][mode].append(run_block(e[0], block, e[2], mode == "pipelined") * 1e6)
        for arm, e in engines.items():
            row = {"entities": n, "arm": arm, "build_s": round(e[4], 3), "specialised": e[0].generic_specialised()}
            for mode in ("sync", "pipelined"):
                v = sorted(res[arm][mode])
                row[f"{mode}_us_per_tick_median"] = round(v[len(v) // 2], 2)
                row[f"{mode}_us_per_tick_all"] = [round(x, 2) for x in res[arm][mode]]
            rows.append(row)
            e[0].close()
        b, u = rows[-2], rows[-1]
        rows.append({"entities": n, "user_over_builtin_sync": round(u["sync_us_per_tick_median"] / b["sync_us_per_tick_median"], 4),
                     "user_over_builtin_pipelined": round(u["pipelined_us_per_tick_median"] / b["pipelined_us_per_tick_median"], 4)})
    text = "\n".join(json.dumps(r) for r in rows)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
