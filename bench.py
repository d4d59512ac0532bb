#!/usr/bin/env python
"""bench.py — rollback frames/s of the snapshot + checksum + re-simulation hot path.

    python bench.py --gpus N --steps K --warmup W            our arm (CUDA engine through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  the reference's CPU path (oracle port) on host cores
    python bench.py ... --dump-outputs DIR                   also writes what the last timed step returned as DIR/*.npy

Metric (BASELINE.json): "rollback frames/sec at 1M entities x 8-frame window".
One step = one SyncTest tick of the stress-test world at steady state: the request vector
[Load(f-8), Adv, Save, Adv, ..., Save(f), Adv] = 1 LoadGameState + 8 SaveGameState (each with its
desync checksum) + 9 AdvanceFrame (SURVEY.md §3.6), i.e. 9 rollback frames per step.

    e2e          THE HEADLINE: the metric through the synchronous C-ABI call a user makes — one bgr_handle_requests per
                 tick from a compiled caller (tools/e2e_caller.c), host request array in, host checksums out, every tick
                 (`e2e_python_caller`: the same loop driven through ctypes)
    value        device throughput with PIPELINED submits (bgr_submit_requests / bgr_collect, K ticks enqueued back to
                 back, CUDA events on the engine's stream); explains the kernel, not reachable through the reference's
                 synchronous contract
    roofline     the fused kernel against the measured HBM copy bandwidth: pipelined / sync (device trace) / e2e / isolated
    timeline     device-side [first block start, last block end, published] of consecutive launches in both modes
    cpu_baseline the oracle port (faithful restatement of the reference's data structures) on host cores

N > 1 (torchrun): entity-range shards, one engine per GPU.  --scaling weak (default): the workload's entity count PER
GPU; --scaling strong: the workload's entity count split over the GPUs (BASELINE C5: 10M total, d=32).  The cross-shard
checksum fold happens inside the engine (bgr_shard_group_join: result pairs in a shared host segment); torch.distributed /
NCCL is launcher plumbing only (rendezvous, barriers, max over ranks).  Rank 0 verifies the folded checksums against one
unsharded engine (`sharded_parity`).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENTITIES = 1_000_000
CHECK_DISTANCE = 8
MAX_PREDICTION = 9       # ggrs requires check_distance < max_prediction
SEED = 0xB200
WORKLOADS = {
    # name: (entities, check_distance, max_prediction)   BASELINE.md configs
    "stress_1m_d8": (1_000_000, 8, 9),        # the headline metric: 1M entities x 8-frame rollback
    "stress_100k_d8": (100_000, 8, 9),        # C2
    "stress_1m_d16": (1_000_000, 16, 17),     # C3
    "p2p_1m_maxpred8": (1_000_000, 0, 8),     # C4: synthetic 2-peer P2P trace, input_delay 2, seed 0xB200
    "stress_10m_d32": (10_000_000, 32, 33),   # C5
}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def build_world(world, n, d, seed):
    from bevy_ggrs_b200.stress import populate, register_particles, synth_particles
    cols = register_particles(world)
    world.build()
    tf, vel, ttl = synth_particles(n, seed, 300 + d + 100000, 300 + d + 100000)  # nothing despawns inside the run
    populate(world, cols, tf, vel, ttl)
    return cols


def pregenerate_ticks(n_ticks, d, maxp, players=2):
    """Request vectors of a SyncTest session (they do not depend on checksum values unless a
    mismatch occurs, which is checked afterwards); d == 0 selects the synthetic P2P trace (C4)."""
    from bevy_ggrs_b200 import capi
    from bevy_ggrs_b200.session import SAVE, P2PTraceSession, SyncTestSession, count_advances
    sess = SyncTestSession(players, d, maxp, input_delay=2) if d > 0 else P2PTraceSession(players, maxp, 2, seed=SEED)
    ticks = []
    for t in range(n_ticks):
        for h in range(players):
            sess.add_local_input(h, (1 << 5) if (t + h) % 3 == 0 else 0)  # INPUT_NOOP schedule
        reqs = sess.advance_frame()
        for r in reqs:
            if r.kind == SAVE:
                sess.save_cell(r.frame, 0)
        ticks.append((capi.make_requests(reqs), len(reqs), count_advances(reqs), capi.make_session_info(sess.info()),
                      [r.frame for r in reqs if r.kind == SAVE]))
    return ticks


def check_synctest_consistency(history):
    """SyncTest property: every re-save of a frame reports the checksum first recorded for it."""
    first = {}
    for frame, cs in history:
        if first.setdefault(frame, cs) != cs:
            return False
    return True


# =================================================================================================
# our arm
# =================================================================================================
class StdoutGuard:
    """N > 1: NCCL's INFO banner (the driver checks `nranks` in it) is printf'ed to fd 1.  Point fd 1 at stderr for the
    whole run and keep the real stdout for the ONE JSON line."""

    def __init__(self, active):
        self.real = None
        if active:
            sys.stdout.flush()
            self.real = os.dup(1)
            os.dup2(2, 1)

    def emit(self, text):
        if self.real is None:
            print(text, flush=True)
        else:
            sys.stdout.flush()
            os.write(self.real, (text + "\n").encode())


def load_caller():
    """tools/libbgr_e2e_caller.so: the compiled per-tick caller of bgr_handle_requests (tools/e2e_caller.c)."""
    from bevy_ggrs_b200 import capi
    path = os.path.join(ROOT, "tools", "libbgr_e2e_caller.so")
    if not os.path.exists(path):
        import __graft_entry__ as g
        g.build_e2e_caller()
    capi.load_library()
    lib = C.CDLL(path)
    lib.bgr_caller_run_ticks.restype = C.c_int
    lib.bgr_caller_run_ticks.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                         C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(C.c_double), C.c_void_p]
    return lib


class CallerBatch:
    """The ticks of one e2e leg as the flat host arrays the compiled caller walks."""

    def __init__(self, tick_list):
        from bevy_ggrs_b200 import capi
        import numpy as np
        self.n = len(tick_list)
        total = sum(t[1] for t in tick_list)
        self.reqs = (capi.bgr_request * max(1, total))()
        self.infos = (capi.bgr_session_info * max(1, self.n))()
        self.offsets = np.zeros(self.n, dtype=np.uint32)
        self.counts = np.zeros(self.n, dtype=np.uint32)
        o = 0
        for i, (arr, nreq, _, info, _) in enumerate(tick_list):
            C.memmove(C.byref(self.reqs, o * C.sizeof(capi.bgr_request)), arr, nreq * C.sizeof(capi.bgr_request))
            self.infos[i] = info
            self.offsets[i], self.counts[i] = o, nreq
            o += nreq
        self.cap = sum(len(t[4]) for t in tick_list) + 8
        self.out = (capi.bgr_checksum * self.cap)()
        self.out_counts = np.zeros(self.n, dtype=np.uint32)
        self.per_tick = np.zeros(self.n, dtype=np.float64)

    def run(self, caller, eng):
        from bevy_ggrs_b200 import capi
        total = C.c_double()
        st = caller.bgr_caller_run_ticks(eng._h, self.infos, self.reqs, self.offsets.ctypes.data, self.counts.ctypes.data,
                                         self.n, self.out, self.cap, self.out_counts.ctypes.data, C.byref(total),
                                         self.per_tick.ctypes.data)
        if st != 0:
            raise RuntimeError(capi.load_library().bgr_last_error().decode())
        return total.value

    def checksums(self):
        k = int(self.out_counts.sum())
        return [(self.out[i].frame, (self.out[i].hi << 64) | self.out[i].lo) for i in range(k)]


def trace_stats(tr):
    """(n, 2) [first block start, last block end] ns per launch -> period / duration / overlap with the next launch."""
    import numpy as np
    if tr.shape[0] < 3:
        return None
    s, e = tr[:, 0].astype(np.int64), tr[:, 1].astype(np.int64)
    pub = (tr[:, 2].astype(np.int64) - e) / 1e3   # last block done -> results + completion word written
    dur = (e - s) / 1e3
    period = np.diff(s) / 1e3
    overlap = (e[:-1] - s[1:]) / 1e3          # > 0: the next launch's first block started before this launch's last block ended
    return {"launches": int(tr.shape[0]), "kernel_us_median": float(np.median(dur)), "period_us_median": float(np.median(period)),
            "overlap_us_median": float(np.median(overlap)), "overlapping_launches": int((overlap > 0).sum()),
            "publish_us_median": float(np.median(pub))}


def run_ours(args):
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        # before torch / NCCL are loaded: the communicator's INIT banner ("... rank r nranks N ...") must stay
        # reachable — on stderr, see StdoutGuard — so that the rank count of a multi-GPU run can be checked
        # (the image exports NCCL_DEBUG=VERSION, which prints no rank count: raise it to INFO / INIT unless the caller
        # asked for something specific through BENCH_NCCL_DEBUG)
        want = os.environ.get("BENCH_NCCL_DEBUG")
        if want:
            os.environ["NCCL_DEBUG"] = want
        elif os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION", "WARN"):
            os.environ["NCCL_DEBUG"] = "INFO"
            os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
        if os.environ.get("RANK", "0") == "0":
            print(f"[bench] NCCL_DEBUG={os.environ.get('NCCL_DEBUG')} NCCL_DEBUG_SUBSYS={os.environ.get('NCCL_DEBUG_SUBSYS')}", file=sys.stderr, flush=True)
    import numpy as np
    import torch
    import torch.distributed as dist
    from bevy_ggrs_b200 import capi
    from bevy_ggrs_b200.engine import Engine
    from bevy_ggrs_b200.sharded import shard_range

    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world_size != args.gpus and world_size > 1:
        args.gpus = world_size
    sharded = world_size > 1
    guard = StdoutGuard(sharded)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if sharded:
        # the communicator is only the launcher-side plumbing (rendezvous, barriers, max-over-ranks of the timings);
        # its INIT banner stays reachable on stderr so that the rank count can be checked
        dist.init_process_group("nccl", device_id=dev)

    n_total, d, maxp = WORKLOADS[args.workload]
    if args.entities:
        n_total = args.entities
    strong = args.scaling == "strong"
    if strong:
        first_row, n = shard_range(n_total, rank, world_size)
        shard_rows = [shard_range(n_total, r, world_size)[1] for r in range(world_size)]
    else:
        n, first_row = n_total, rank * n_total          # weak scaling: the workload's entity count PER GPU
        shard_rows = [n_total] * world_size
    K, W = args.steps, max(3, args.warmup)
    eng = Engine(max_entities=n, max_depth=maxp, fps=60, device=local_rank,
                 flags=capi.BGR_CFG_SHARDED if sharded else 0, order_base=first_row)
    # started long before the timed region: nvidia-smi's start-up and first polls slow a 2 ms region by ~1 %
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    cols = build_world(eng, n, d, SEED + rank)
    stream = torch.cuda.ExternalStream(eng.stream(), device=dev)   # the stream the kernels are launched on
    slot_bytes = eng.slot_bytes()
    if sharded:
        # the cross-shard checksum exchange happens INSIDE the engine from here on (bgr_shard_group_join): every
        # bgr_collect / bgr_handle_requests returns the whole world's frame checksum; no torch call per tick
        names = [f"bgr_bench_{os.getpid()}_{int(time.time() * 1e6)}" if rank == 0 else None]
        dist.broadcast_object_list(names, src=0)
        eng.shard_group_join(names[0], rank, world_size, 120000)

    fill = max(d, maxp) + 2           # ticks until the request vector has its steady-state shape
    K2 = min(K, 500) if world_size == 1 else 0   # ticks of the host-mirror leg (N = 1 only)
    BT = int(os.environ.get("BENCH_BATCH_TICKS", "4")) if world_size == 1 and d > 0 else 0   # catch-up leg: ticks per request vector
    BT = min(BT, capi.BGR_MAX_REQUESTS // (2 * d + 2)) if d > 0 else 0                          # ... that fit one call
    K3 = (min(K, 400) // BT) * BT if BT > 1 else 0
    KT = 64                            # ticks of each traced leg (pipelined / synchronous)
    ticks = pregenerate_ticks(fill + W + 3 * K + K2 + K3 + 2 * KT, d, maxp)
    pos = [0]

    def take(k):
        out = ticks[pos[0]: pos[0] + k]
        pos[0] += k
        return out

    history = []
    depth = 4 if sharded else 2     # un-collected submits kept queued on the GPU (hides the host loop / rank jitter)

    def run_pipelined(tick_list):
        """Returns the checksums bgr_collect handed back for the last tick."""
        inflight, last = 0, []
        for arr, nreq, _, info, _ in tick_list:
            eng.submit_prepared(info, arr, nreq)
            inflight += 1
            if inflight > depth:
                last = eng.collect()
                history.extend(last)
                inflight -= 1
        while inflight:
            last = eng.collect()
            history.extend(last)
            inflight -= 1
        return last

    def barrier():
        torch.cuda.synchronize()
        if sharded:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if not sharded:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    caller = load_caller()
    lib = capi.load_library()

    run_pipelined(take(fill + W))           # ring fill + warm-up (>= 3 steady-state ticks)
    barrier()
    # ---------------- value: device-timed, K ticks back to back ----------------
    sampler.rows.clear()              # clocks of the timed legs only
    timed = take(K)
    l0 = eng.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    last_checksums = run_pipelined(timed)
    ev1.record(stream)
    barrier()
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    launches = eng.launch_count() - l0
    adv_total = sum(t[2] for t in timed)
    adv_per_tick = adv_total / K
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, cols, last_checksums)
    # ---------------- e2e: ONE synchronous bgr_handle_requests per tick, host arrays in / host checksums out ----------------
    e2e_ticks = take(K)
    batch = CallerBatch(e2e_ticks)
    barrier()
    e2e_s = max_over_ranks(batch.run(caller, eng))
    history.extend(batch.checksums())
    clocks = sampler.stop() if rank == 0 else None
    e2e_p50_us = float(np.median(batch.per_tick) * 1e6)
    h2d = sum(C.sizeof(capi.bgr_request) * t[1] + C.sizeof(capi.bgr_session_info) for t in e2e_ticks) / K
    d2h = sum(64 * len(t[4]) + 8 for t in e2e_ticks) / K  # one 8 x u64 result row per SaveGameState + the completion word, pinned host memory
    # the same loop driven from Python through ctypes (what round 1 reported as e2e)
    py_ticks = take(K)
    out = (capi.bgr_checksum * capi.BGR_MAX_REQUESTS)()
    nout = C.c_uint32()
    barrier()
    t0 = time.perf_counter()
    for arr, nreq, _, info, _ in py_ticks:
        st = lib.bgr_handle_requests(eng._h, C.byref(info), arr, nreq, out, capi.BGR_MAX_REQUESTS, C.byref(nout))
        if st != 0:
            raise RuntimeError(lib.bgr_last_error().decode())
        history.extend((out[i].frame, (out[i].hi << 64) | out[i].lo) for i in range(nout.value))
    e2e_py_s = max_over_ranks(time.perf_counter() - t0)

    # ---------------- device-side timeline of both modes (bgr_trace_enable; NOT part of the timed regions above) ----------------
    timeline = {}
    sync_kernel_s = sync_bytes = None
    try:
        eng.trace_enable(2 * KT + 8)
        tp = take(KT)
        run_pipelined(tp)
        barrier()
        tr_p = eng.trace_read(2 * KT + 8)
        tb_ticks = take(KT)
        tb = CallerBatch(tb_ticks)
        tb.run(caller, eng)
        history.extend(tb.checksums())
        tr_all = eng.trace_read(2 * KT + 8)
        tr_s = tr_all[tr_p.shape[0]:]
        eng.trace_enable(0)
        # synchronous launches: bytes and device time summed over the SAME ticks (request vectors of a P2P trace differ in size)
        if tr_s.shape[0] == len(tb_ticks):
            sync_kernel_s = float((tr_s[:, 1].astype(np.int64) - tr_s[:, 0].astype(np.int64)).sum()) * 1e-9
            sync_bytes = float(sum(len(t[4]) + 2 for t in tb_ticks)) * slot_bytes
        timeline = {"pipelined": trace_stats(tr_p), "synchronous": trace_stats(tr_s),
                    "note": "GPU globaltimer, first block start .. last block end of every fused launch; "
                            "overlap > 0 = the next tick's first wave ran inside this tick's tail (tile dependencies)"}
        if args.trace_out and rank == 0:
            with open(args.trace_out, "w") as f:
                f.write("mode,launch,first_block_start_ns,last_block_end_ns,published_ns\n")
                for mode, tr in (("pipelined", tr_p), ("synchronous", tr_s)):
                    base = int(tr[0, 0]) if tr.shape[0] else 0
                    for i in range(tr.shape[0]):
                        f.write(f"{mode},{i},{int(tr[i, 0]) - base},{int(tr[i, 1]) - base},{int(tr[i, 2]) - base}\n")
    except Exception as exc:  # an optional leg must not cost the headline line
        timeline = {"error": repr(exc)}

    # ---------------- e2e with a host mirror: every tick also downloads Transform.translation ----------------
    # What a host-resident ECS needs back per tick to draw the particles (INTEGRATION.md "mirror"): 12 B/entity
    # packed on the GPU, copied D2H on a copy stream into page-locked memory while the next tick runs.
    def mirror_leg():
        m_ticks = take(K2)
        bufs = [eng.host_alloc(n, 12), eng.host_alloc(n, 12)]
        pending = None
        barrier()
        t0 = time.perf_counter()
        for i, (arr, nreq, _, info, _) in enumerate(m_ticks):
            eng.submit_prepared(info, arr, nreq)
            tk = eng.download_begin(0, 0, 12, 0, n, bufs[i & 1])
            history.extend(eng.collect())
            if pending is not None:
                eng.download_wait(pending)   # the previous tick's mirror is now readable on the host
            pending = tk
        eng.download_wait(pending)
        m_s = time.perf_counter() - t0
        return {"value": sum(t[2] for t in m_ticks) / m_s, "unit": "rollback frames/s", "ticks": K2,
                "d2h_bytes_per_step": 12 * n + sum(64 * len(t[4]) + 8 for t in m_ticks) / K2,
                "d2h_gbs": 12 * n * K2 / m_s / 1e9,
                "note": "e2e + bgr_download_begin/wait of Transform.translation (12 B/entity) every tick, "
                        "double-buffered pinned host memory; PCIe-bound when 12 B x entities / tick exceeds the link"}

    mirror = None
    if K2:
        try:
            mirror = mirror_leg()
        except Exception as exc:
            mirror = {"error": repr(exc)}

    def batch_leg():
        # catch-up shape of run_ggrs_schedules' inner loop (schedule_systems.rs:60-82): several ticks' request
        # vectors handed over in one call
        b_ticks = take(K3)
        groups = []
        for g in range(0, K3, BT):
            grp = b_ticks[g:g + BT]
            n_req = sum(t[1] for t in grp)
            arr = (capi.bgr_request * n_req)()
            o = 0
            for t in grp:
                for i in range(t[1]):
                    arr[o] = t[0][i]
                    o += 1
            groups.append((arr, n_req, sum(t[2] for t in grp), grp[0][3], None))
        barrier()
        evb0, evb1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        lb0 = eng.launch_count()
        evb0.record(stream)
        run_pipelined(groups)
        evb1.record(stream)
        barrier()
        bms = evb0.elapsed_time(evb1)
        return {"ticks_per_call": BT, "value": sum(g[2] for g in groups) / (bms * 1e-3), "unit": "rollback frames/s",
                "ms_per_tick": bms / K3, "gpu_launches": eng.launch_count() - lb0, "fused": bool(eng.last_path_fused()),
                "note": "NOT the headline: several ticks' request vectors per bgr_handle_requests call (the catch-up "
                        "shape of run_ggrs_schedules' inner loop); one launch per call, the live image is written "
                        "once per call"}

    batched = None
    if K3:
        try:
            batched = batch_leg()
        except Exception as exc:
            batched = {"error": repr(exc)}

    consistent = check_synctest_consistency(history)
    fused = eng.last_path_fused()

    # ---------------- N > 1: the folded checksums against ONE engine holding the whole population ----------------
    sharded_parity = None
    if sharded:
        barrier()
        ok = 1
        if rank == 0:
            try:
                sharded_parity = verify_against_unsharded(shard_rows, d, maxp, local_rank, ticks[:fill + 3], history)
                ok = 1 if sharded_parity["equal"] else 0
            except Exception as exc:
                sharded_parity = {"error": repr(exc)}
                ok = 0
        t = torch.tensor([ok], device=dev, dtype=torch.int32)
        dist.broadcast(t, src=0)
        consistent = consistent and bool(t.item())

    # ---------------- roofline of the dominant (only) kernel ----------------
    ms_per_step = ms / K
    # per tick: read 1 image (slot or live) + write one slot per Save + write the live image (DESIGN.md §Roofline)
    alg_bytes = sum(len(t[4]) + 2 for t in timed) / K * slot_bytes
    achieved = alg_bytes / (ms_per_step * 1e-3) / 1e9
    # SURVEY §8(d)'s other accounting, for reference: what the reference's UNFUSED schedule would move for the same
    # requests (every Save and Load = read + write of an image, every Advance = 64 B/entity); it exceeds the HBM
    # peak because the fused kernel never moves those bytes
    n_loads = sum(1 for t in timed for i in range(t[1]) if t[0][i].kind == capi.BGR_REQ_LOAD)
    unfused_bytes = (sum(2 * len(t[4]) for t in timed) + 2 * n_loads) / K * slot_bytes + 64.0 * n * adv_per_tick
    achieved_unfused = unfused_bytes / (ms_per_step * 1e-3) / 1e9
    peak, peak_src = measured_hbm_peak()
    traffic = isolated = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            traffic = tj.get(args.workload)
            isolated = tj.get("isolated_launch_us", {}).get(args.workload)
        except Exception:
            traffic = None
    e2e_alg = sum(len(t[4]) + 2 for t in e2e_ticks) / K * slot_bytes
    sync_kernel_us = (timeline.get("synchronous") or {}).get("kernel_us_median")

    # ---------------- CPU baseline (rank 0, N == 1 only): oracle port on host cores ----------------
    cpu = cpu_soa = None
    if rank == 0 and world_size == 1 and not args.no_cpu_baseline:
        cpu = run_cpu_sample(n, d, maxp, rollback_ticks=4, warm_ticks=1)   # the first rollback tick (cold hash maps) is not timed
        if d > 0:
            cpu_soa = run_cpu_soa_sample(n, d, maxp)
    snap = snap10 = skip = None
    if rank == 0 and world_size == 1 and not args.no_snapshot_bench:
        eng.close()
        snap = snapshot_bench(n, maxp, local_rank)
        try:
            snap10 = snapshot_bench(10_000_000, maxp, local_rank, iters=20)   # 610 MB images: out of L2, an HBM measurement
        except Exception as exc:
            snap10 = {"error": repr(exc)}
        skip = skip_unchanged_bench(n, d, maxp, local_rank, ticks, fill, W, K, history)
    generic = None
    if rank == 0 and world_size == 1 and not args.no_snapshot_bench:
        try:
            generic = generic_world_leg(n)
        except Exception as exc:  # an optional leg must not cost the headline line
            generic = {"error": repr(exc)}

    if rank == 0:
        value = sum(shard_rows) / n_total * adv_total / (ms * 1e-3) if strong else world_size * adv_total / (ms * 1e-3)
        scale = (sum(shard_rows) / n_total) if strong else world_size
        e2e_value = scale * sum(t[2] for t in e2e_ticks) / e2e_s
        line = {
            "metric": "rollback frames/sec at 1M entities x 8-frame window (SyncTest: 1 Load + 8 Save+checksum + 9 Advance per tick)",
            "value": value, "unit": "rollback frames/s", "n_gpus": world_size, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "u64 (seahash) + f32 (particles, no FMA) + u8 copy", "data": "synthetic (numpy PCG64 seed 0xB200; BASELINE.md shapes)",
            "config": {"workload": args.workload, "entities_per_gpu": n, "entities_total": sum(shard_rows), "check_distance": d,
                       "max_prediction": maxp,
                       "columns": "Transform40+Velocity12+Ttl8+alive1 = 61 B/entity/slot", "checksum": "every saved frame",
                       "advances_per_step": adv_per_tick,
                       "l2": "inputs larger than L2: each tick reads 1 slot and writes 9 images of "
                       f"{slot_bytes/1e6:.0f} MB (ring {maxp} slots)", "path": "fused" if fused else "stepwise",
                       "value_is": "device-timed PIPELINED submits (bgr_submit_requests / bgr_collect, consecutive launches overlap); "
                                   "the synchronous per-tick contract of the reference is `e2e`",
                       "sharding": (f"entity-range x{world_size}; cross-shard checksum fold inside the engine "
                                    "(bgr_shard_group_join: kernels store their 64 B partial rows into a shared host segment, "
                                    "every rank's CPU polls and folds; no collective call per tick)") if sharded else "none"},
            "gpu_launches": launches,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "rollback frames/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_s / K * 1e3, "p50_us_per_call": e2e_p50_us,
                    "caller": "compiled (tools/e2e_caller.c): one synchronous bgr_handle_requests per tick",
                    "note": "request vector from host memory, checksums to host memory, every tick; "
                            "component columns live in HBM by design and never cross"},
            "e2e_python_caller": {"value": scale * sum(t[2] for t in py_ticks) / e2e_py_s, "unit": "rollback frames/s",
                                  "note": "the same per-tick call driven from Python through ctypes (round 1's e2e)"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic,
                         "traffic_source": "constant: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture "
                                           "(profiles/traffic.json), NOT measured in this run",
                         "peak_source": peak_src, "kernel": "k_particles_program",
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "pipelined": {"achieved": achieved, "frac": achieved / peak,
                                       "how": "algorithmic bytes / (CUDA-event time of K back-to-back launches / K); launches overlap"},
                         "sync": None if not sync_kernel_s else {
                             "kernel_us": sync_kernel_us, "achieved": sync_bytes / sync_kernel_s / 1e9,
                             "frac": sync_bytes / sync_kernel_s / 1e9 / peak,
                             "how": "algorithmic bytes / device duration (first block start .. last block end, globaltimer), both "
                                    f"summed over the launches of {KT} synchronous bgr_handle_requests calls; kernel_us = the median launch"},
                         "e2e": {"achieved": e2e_alg / (e2e_s / K) / 1e9, "frac": e2e_alg / (e2e_s / K) / 1e9 / peak,
                                 "how": "algorithmic bytes / host wall time per synchronous call"},
                         "isolated": None if not isolated else {
                             "kernel_us": isolated, "frac": alg_bytes / (isolated * 1e-6) / 1e9 / peak,
                             "how": "constant: ncu gpu__time_duration of one serialised cold-cache launch (profiles/traffic.json)"},
                         "unfused_accounting": {"bytes_per_step": unfused_bytes, "effective_gbs": achieved_unfused,
                                                "note": "bytes the reference's one-schedule-per-request path would move "
                                                        "(2S per Save/Load + 64 B per Advance per entity); not a roofline claim"}},
            "timeline": timeline,
            "synctest_consistent": consistent,
        }
        if sharded_parity is not None:
            line["sharded_parity"] = sharded_parity
        if cpu:
            line["cpu_baseline"] = cpu
        if cpu_soa:
            line["cpu_baseline_optimised_soa"] = cpu_soa
        if mirror:
            line["e2e_host_mirror"] = mirror
        if batched:
            line["catch_up_batch"] = batched
        if snap:
            line["snapshot_save_restore"] = snap
        if snap10:
            line["snapshot_save_restore_10m"] = snap10
        if skip:
            line["opt_in_skip_unchanged_planes"] = skip
        if generic:
            line["generic_world"] = generic
        guard.emit(json.dumps(line))
    eng.close()
    if sharded:
        dist.barrier()
        dist.destroy_process_group()
    if not consistent:
        sys.exit(3)


DUMP_SAMPLE_ROWS = 1 << 18   # 72 B per sampled row across the dumped arrays: 19 MB at most


def dump_outputs(out_dir, eng, cols, checksums):
    """What the timed path handed back on its last step, as float arrays two builds can be compared with: the
    (frame, checksum) pairs bgr_collect returned, and the live particle columns of a fixed, seeded sample of rows."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    rows_total = eng.row_count()
    rows = np.sort(np.random.default_rng(SEED).choice(rows_total, size=min(rows_total, DUMP_SAMPLE_ROWS), replace=False))
    t, v, l = cols
    arrays = {
        # frame, then the u128 checksum as four u32 words, least significant first (each exact in float64)
        "checksums": np.array([[f] + [(c >> s) & 0xFFFFFFFF for s in (0, 32, 64, 96)] for f, c in checksums],
                              dtype=np.float64).reshape(-1, 5),
        "sample_rows": rows.astype(np.float64),
        "alive": eng.read_alive(0, rows_total)[rows].astype(np.float32),
        "transform": eng.read_component(t, 0, rows_total)[rows].view(np.float32),          # translation | rotation | scale
        "velocity": eng.read_component(v, 0, rows_total)[rows].view(np.float32),
        "ttl": eng.read_component(l, 0, rows_total)[rows].view(np.uint64)[:, 0].astype(np.float64),
    }
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def generic_world_leg(n):
    """A registration that is NOT the particles bundle (optional Score / Health + a 12-byte Tag, all checksummed, two u32
    systems; scripts/generic_world_bench.py) at the headline entity count, synchronous SyncTest ticks (check_distance 8) driven
    from Python: once on the kernel bgr_build compiled for it with NVRTC, once on the precompiled interpreter kernel."""
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import generic_world_bench as g
    out = {"entities": n, "check_distance": 8, "world": "Score 4 B optional + Health 4 B optional (satsub-despawn) + Tag 12 B, all checksummed",
           "note": "synchronous ticks from Python; kernel_us = device globaltimer, first block start .. last block end (median)"}
    old = os.environ.get("BGR_TUNE_JIT")
    try:
        for name, jit in (("specialised_kernel", "2"), ("interpreter_kernel", "0")):
            os.environ["BGR_TUNE_JIT"] = jit
            w = g.presence_world(n, 0)
            try:
                out[name] = g.run(w, 100)
            finally:
                w.close()
    finally:
        if old is None:
            os.environ.pop("BGR_TUNE_JIT", None)
        else:
            os.environ["BGR_TUNE_JIT"] = old
    return out


def verify_against_unsharded(shard_rows, d, maxp, device_index, tick_list, history):
    """Rank 0, N > 1: run the first ticks on ONE engine that holds every shard's population (order_base 0) and compare
    its checksums, frame by frame, with what the sharded engines folded — parity of the multi-GPU path on hardware."""
    import numpy as np
    from bevy_ggrs_b200.engine import Engine
    from bevy_ggrs_b200.stress import populate, register_particles, synth_particles
    total = sum(shard_rows)
    ref = Engine(max_entities=total, max_depth=maxp, fps=60, device=device_index)
    cols = register_particles(ref)
    ref.build()
    for r, rows in enumerate(shard_rows):
        tf, vel, ttl = synth_particles(rows, SEED + r, 300 + d + 100000, 300 + d + 100000)
        populate(ref, cols, tf, vel, ttl)
    got = {}
    for f, c in history:
        got.setdefault(f, c)
    n_frames, equal = 0, True
    for arr, nreq, _, info, _ in tick_list:
        ref.submit_prepared(info, arr, nreq)
        for f, c in ref.collect():
            n_frames += 1
            equal = equal and (got.get(f) == c)
    ref.close()
    return {"equal": bool(equal), "ticks": len(tick_list), "checksums_compared": n_frames, "entities": total,
            "how": "rank 0 re-ran the first ticks on one unsharded engine holding every shard's population; "
                   "every frame checksum must equal the cross-shard fold"}


def skip_unchanged_bench(n, d, maxp, device_index, ticks, fill, W, K, reference_history):
    """Same workload with BGR_CFG_SKIP_UNCHANGED_PLANES (opt-in, NOT the headline): planes no registered system
    writes (Transform.rotation/scale, 28 of 61 B/entity) are not rewritten into slots that already hold them.
    Every checksum must equal the default run's.  Bytes are counted as actually moved: 33 B/entity/image."""
    import torch
    from bevy_ggrs_b200 import capi
    from bevy_ggrs_b200.engine import Engine
    eng = Engine(max_entities=n, max_depth=maxp, fps=60, device=device_index, flags=capi.BGR_CFG_SKIP_UNCHANGED_PLANES)
    build_world(eng, n, d, SEED)
    stream = torch.cuda.ExternalStream(eng.stream())
    hist = []

    def run(tl):
        inflight = 0
        for arr, nreq, _, info, _ in tl:
            eng.submit_prepared(info, arr, nreq)
            inflight += 1
            if inflight > 2:
                hist.extend(eng.collect()); inflight -= 1
        while inflight:
            hist.extend(eng.collect()); inflight -= 1

    with torch.cuda.stream(stream):
        run(ticks[:fill + W])
        torch.cuda.synchronize()
        timed = ticks[fill + W: fill + W + K]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        run(timed)
        e1.record(stream)
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    rows = eng.row_count()
    eng.close()
    ref = {}
    for f, c in reference_history:
        ref.setdefault(f, c)
    same = all(ref.get(f, c) == c for f, c in hist)
    moved = sum(len(t[4]) + 2 for t in timed) / K * rows * 33
    peak, _ = measured_hbm_peak()
    return {"value": sum(t[2] for t in timed) / (ms * 1e-3), "unit": "rollback frames/s", "ms_per_step": ms / K,
            "checksums_equal_default_run": same, "bytes_moved_per_step": moved,
            "achieved_gbps": moved / (ms / K * 1e-3) / 1e9, "frac_of_measured_hbm": moved / (ms / K * 1e-3) / 1e9 / peak,
            "note": "opt-in BGR_CFG_SKIP_UNCHANGED_PLANES: redundant stores of planes no system writes are elided "
                    "(content-version tracking); NOT used for the headline value"}


def snapshot_bench(n, maxp, device_index, iters=50):
    """M2 of BASELINE.md: snapshot save + restore GB/s = 4*S*E / (t_save + t_load), one request per launch.
    Two implementations of the same C-ABI calls are timed: the fused program kernel with a one-op
    program, and the TMA-staged (cp.async.bulk) image copy of the stepwise path."""
    import torch
    from bevy_ggrs_b200 import capi
    from bevy_ggrs_b200.engine import Engine
    from bevy_ggrs_b200.session import LOAD, SAVE, Request
    out = {}
    peak, _ = measured_hbm_peak()
    for name, flags in (("fused_program", 0), ("tma_bulk_copy", capi.BGR_CFG_FORCE_STEPWISE)):
        eng = Engine(max_entities=n, max_depth=2, fps=60, device=device_index, flags=flags)
        build_world(eng, n, 8, SEED)
        stream = torch.cuda.ExternalStream(eng.stream())
        info = capi.make_session_info((0, 0, 0, 0))
        save = capi.make_requests([Request(SAVE, 0)])
        load = capi.make_requests([Request(LOAD, 0)])
        res = {}
        with torch.cuda.stream(stream):
            for label, arr in (("save", save), ("load", load)):
                for _ in range(5):
                    eng.submit_prepared(info, arr, 1); eng.collect()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                inflight = 0
                for _ in range(iters):
                    eng.submit_prepared(info, arr, 1)
                    inflight += 1
                    if inflight > 2:
                        eng.collect(); inflight -= 1
                while inflight:
                    eng.collect(); inflight -= 1
                e1.record(stream)
                torch.cuda.synchronize()
                res[label + "_us"] = e0.elapsed_time(e1) * 1e3 / iters
        sb = eng.slot_bytes()
        gbps = 4 * sb / ((res["save_us"] + res["load_us"]) * 1e-6) / 1e9
        res.update({"gb_per_s": gbps, "frac_of_measured_hbm": gbps / peak, "slot_bytes": sb,
                    "note": "2*S*E bytes per save (with checksum) and per load; 61 MB images fit L2 (126 MB): see ncu dram bytes"})
        out[name] = res
        eng.close()
    return out


# =================================================================================================
# the reference's CPU path (oracle port) — test infrastructure timed as the baseline
# =================================================================================================
def run_cpu_sample(n, d, maxp, rollback_ticks, entities=None, warm_ticks=0):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_backend import OracleWorld
    from bevy_ggrs_b200.session import SAVE, SyncTestSession, count_advances
    e = entities or n
    threads = max(1, min(os.cpu_count() or 1, 8))
    orc = OracleWorld(fps=60, save_threads=threads)
    build_world(orc, e, d, SEED)
    sess = SyncTestSession(2, d, maxp, input_delay=2)
    total_ns, total_adv, timed = 0, 0, 0
    t = 0
    while timed < rollback_ticks:
        for h in range(2):
            sess.add_local_input(h, (1 << 5) if (t + h) % 3 == 0 else 0)
        reqs = sess.advance_frame()
        cs = orc.handle_requests(sess.info(), reqs)
        for frame, c in cs:
            sess.save_cell(frame, c)
        if reqs[0].kind == 1:  # steady-state rollback tick
            if warm_ticks > 0:
                warm_ticks -= 1
            else:
                total_ns += orc.last_elapsed_ns
                total_adv += count_advances(reqs)
                timed += 1
        t += 1
    orc.close()
    fps = total_adv / (total_ns * 1e-9)
    scaled = fps * (e / n)
    return {"value": scaled, "unit": "rollback frames/s", "cores": threads, "kind": "port",
            "sample": f"{timed} steady-state SyncTest ticks (d={d}) of the oracle port at {e} entities"
                      + ("" if e == n else f", scaled by {e}/{n} to the {n}-entity metric")
                      + "; per-type save/checksum systems overlapped on the stated cores like Bevy's multithreaded executor, "
                        "AdvanceWorld single-threaded (lib.rs:237)",
            "seconds_per_tick": total_ns * 1e-9 / timed}


def run_cpu_soa_sample(n, d, maxp, rollback_ticks=12):
    """The optimised CPU SoA bar (BASELINE.md §2(2), oracle/soa_baseline.hpp): flat columns, memcpy slots, the
    request vector executed per entity range on every host core.  An honesty check beside the faithful port."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_backend import SoaWorld
    from bevy_ggrs_b200.session import SyncTestSession, count_advances
    from bevy_ggrs_b200.stress import synth_particles
    tf, vel, ttl = synth_particles(n, SEED, 300 + d + 100000, 300 + d + 100000)
    threads = os.cpu_count() or 1
    soa = SoaWorld(tf, vel, ttl, depth=maxp, threads=threads)
    sess = SyncTestSession(2, d, maxp, input_delay=2)
    per_tick, timed, t, adv = [], 0, 0, 0
    while timed < rollback_ticks + 2:
        for h in range(2):
            sess.add_local_input(h, (1 << 5) if (t + h) % 3 == 0 else 0)
        reqs = sess.advance_frame()
        for frame, c in soa.handle_requests(sess.info(), reqs):
            sess.save_cell(frame, c)
        if reqs[0].kind == 1:
            if timed > 1:  # first two rollback ticks = warm-up (thread pool, page faults of the slot ring)
                per_tick.append(soa.last_elapsed_ns * 1e-9)
                adv = count_advances(reqs)
            timed += 1
        t += 1
    soa.close()
    med = statistics.median(per_tick)   # all-core runs are noisy on a shared host: the median tick, not the mean
    return {"value": adv / med, "unit": "rollback frames/s", "cores": threads, "kind": "port-optimised-soa",
            "sample": f"median of {rollback_ticks} steady-state SyncTest ticks (d={d}) at {n} entities, flat SoA columns + memcpy slots + "
                      f"per-range threads on all {threads} host cores (NOT the reference's data structures)",
            "seconds_per_tick": med, "seconds_per_tick_min_max": [min(per_tick), max(per_tick)]}


def try_real_reference(n, d, ticks, seed):
    """BASELINE.md §2(3): where a Rust toolchain and a bevy_ggrs checkout named by BEVY_GGRS_PATH exist (probed at run
    time), build oracle/ref_harness against the UNMODIFIED reference crate and time the real Bevy SyncTest path.
    Returns the harness' timing dict or None."""
    import shutil
    import tempfile
    ref = os.environ.get("BEVY_GGRS_PATH", "")
    if not ref or not shutil.which("cargo") or not os.path.exists(os.path.join(ref, "Cargo.toml")):
        return None
    try:
        tmp = tempfile.mkdtemp()
        shutil.copytree(os.path.join(ROOT, "oracle", "ref_harness"), os.path.join(tmp, "harness"))
        man = os.path.join(tmp, "harness", "Cargo.toml")
        open(man, "w").write(open(man).read().replace('path = "../../../reference"', f'path = "{ref}"'))
        subprocess.run([sys.executable, os.path.join(ROOT, "tests", "golden", "gen_reference_inputs.py"),
                        os.path.join(tmp, "p.bin"), str(n), hex(seed), str(300 + d + 100000), str(300 + d + 100000)], check=True)
        r = subprocess.run(["cargo", "run", "--release", "--quiet", "--manifest-path", man, "--",
                            os.path.join(tmp, "p.bin"), str(n), str(d), str(ticks)], capture_output=True, text=True, timeout=1500)
        if r.returncode != 0:
            return None
        return json.loads(r.stdout)["timing"]
    except Exception:
        return None


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n, d, maxp = WORKLOADS[args.workload]
    K, W = args.steps, args.warmup
    real = try_real_reference(min(n, 200_000), d, d + 2 + K + W, SEED) if d > 0 else None
    if real:  # the unmodified crate ran here: report it (scaled linearly to the metric's entity count — flatters the CPU)
        e = min(n, 200_000)
        v = real["rollback_frames_per_s"] * (e / n)
        line = {"impl": "reference", "metric": "rollback frames/sec at 1M entities x 8-frame window (SyncTest: 1 Load + 8 Save+checksum + 9 Advance per tick)",
                "value": v, "unit": "rollback frames/s", "n_gpus": args.gpus, "steps": K, "warmup": W,
                "ms_per_step": real["seconds"] / max(1, real["ticks"]) * 1e3 * (n / e), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u64 (seahash) + f32 + bytes", "data": "synthetic (same generator and seed as the GPU arm)",
                "config": {"workload": args.workload, "entities_per_gpu": n, "check_distance": d, "max_prediction": maxp,
                           "note": f"the UNMODIFIED bevy_ggrs crate through oracle/ref_harness (headless Bevy app), {e} entities "
                                   f"scaled by {e}/{n}"},
                "cpu_baseline": {"value": v, "unit": "rollback frames/s", "cores": 1, "kind": "reference",
                                 "sample": f"{real['ticks']} SyncTest ticks at {e} entities of the real crate"},
                "e2e": {"value": v, "unit": "rollback frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return
    # bound the whole run to a few minutes: the port needs ~2.6 s per 1M-entity rollback tick with 8 threads and
    # about linear time in the entity count (super-linear in reality — hash maps fall out of cache — so a smaller
    # sample flatters the CPU, never the GPU); d+1 plain ticks fill the ring before the first rollback tick
    budget_s = 120.0
    per_tick_1m = 2.6 * (n / 1_000_000)
    est = per_tick_1m * (K + W + d + 1)
    e = n if est <= budget_s else max(10_000, int(n * budget_s / est) // 1000 * 1000)
    r = run_cpu_sample(n, d, maxp, rollback_ticks=K, entities=e, warm_ticks=W)
    line = {
        "impl": "reference",
        "metric": "rollback frames/sec at 1M entities x 8-frame window (SyncTest: 1 Load + 8 Save+checksum + 9 Advance per tick)",
        "value": r["value"], "unit": "rollback frames/s", "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": r["seconds_per_tick"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64 (seahash) + f32 + bytes", "data": "synthetic (same generator and seed as the GPU arm)",
        "config": {"workload": args.workload, "entities_per_gpu": n, "check_distance": d, "max_prediction": maxp,
                   "note": "no Rust toolchain or bevy_ggrs checkout (BEVY_GGRS_PATH) was found: this arm times the "
                           "oracle port, a faithful CPU restatement of the reference's data structures and loops"},
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": "rollback frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from untouched (it may be read-only)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="stress_1m_d8", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-snapshot-bench", action="store_true")
    ap.add_argument("--entities", type=int, default=0, help="override the workload's entity count (scaling studies)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = the workload's entity count per GPU; strong = the workload's entity count split over the GPUs (BASELINE C5)")
    ap.add_argument("--trace-out", default="", help="write the device-side launch timeline (CSV) here")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the timed path returned on its last step (checksums + a seeded row sample of the "
                         "world) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA arm only")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
