"""CPU checks of bench.py's host-side helpers (no GPU): the flat request arrays the compiled caller walks, the
launch-timeline statistics, and the stdout guard that keeps the one JSON line apart from NCCL's banner."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from bevy_ggrs_b200 import capi  # noqa: E402


def test_caller_batch_flattens_ticks_in_order():
    ticks = bench.pregenerate_ticks(14, 4, 5)
    b = bench.CallerBatch(ticks)
    assert b.n == 14 and list(b.counts) == [t[1] for t in ticks]
    assert list(b.offsets) == list(np.cumsum([0] + [t[1] for t in ticks[:-1]]))
    for i, (arr, nreq, _, info, _) in enumerate(ticks):
        for k in range(nreq):
            r = b.reqs[int(b.offsets[i]) + k]
            assert (r.kind, r.frame, r.n_players, bytes(r.inputs)) == (arr[k].kind, arr[k].frame, arr[k].n_players, bytes(arr[k].inputs))
        assert (b.infos[i].kind, b.infos[i].max_prediction, b.infos[i].check_distance) == (info.kind, info.max_prediction, info.check_distance)
    assert b.cap >= sum(len(t[4]) for t in ticks)
    # steady-state SyncTest tick at d = 4: Load + 4 x Advance + 4 x Save = 9 requests, 5 of them AdvanceFrame
    assert ticks[-1][1] == 10 and ticks[-1][2] == 5 and len(ticks[-1][4]) == 4


def test_trace_stats_reports_overlap_and_publish_time():
    # three launches: the second starts 2 us before the first ends, the third 1 us after the second ends
    tr = np.array([[1000, 11000, 12000, 0], [9000, 20000, 21500, 0], [21000, 30000, 31000, 0]], dtype=np.uint64)
    st = bench.trace_stats(tr)
    assert st["launches"] == 3 and st["overlapping_launches"] == 1
    assert st["kernel_us_median"] == 10.0 and st["period_us_median"] == 10.0
    assert st["publish_us_median"] == 1.0
    assert bench.trace_stats(tr[:2]) is None


def test_stdout_guard_keeps_the_json_line_alone_on_stdout():
    code = ("import os, sys; sys.path.insert(0, %r); import bench\n"
            "g = bench.StdoutGuard(True)\n"
            "os.write(1, b'NCCL INFO comm rank 0 nranks 2\\n')\n"     # what a C library printf's to fd 1
            "print('python noise')\n"
            "g.emit('{\"ok\": 1}')\n") % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.stdout == '{"ok": 1}\n'
    assert "nranks 2" in r.stderr and "python noise" in r.stderr


def test_synctest_consistency_check():
    assert bench.check_synctest_consistency([(1, 5), (2, 6), (1, 5)])
    assert not bench.check_synctest_consistency([(1, 5), (1, 7)])


def test_dump_outputs_is_exact_seeded_and_float(tmp_path, monkeypatch):
    """--dump-outputs on a CPU world of the same shape: u128 checksums survive as float64 words bit for bit, the row
    sample is the same on every run, and every array is float32 or float64."""
    from oracle_backend import OracleWorld
    monkeypatch.setattr(bench, "DUMP_SAMPLE_ROWS", 100)
    orc = OracleWorld(fps=60)
    cols = bench.build_world(orc, 1000, 4, bench.SEED)
    checksums = [(3, (1 << 127) | 0x0123456789ABCDEF), (4, 7)]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), orc, cols, checksums)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["alive.npy", "checksums.npy", "sample_rows.npy", "transform.npy", "ttl.npy", "velocity.npy"]
    got = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    for n in names:
        assert np.array_equal(got[n[:-4]], np.load(tmp_path / "b" / n))
        assert got[n[:-4]].dtype in (np.float32, np.float64)
    assert [(int(r[0]), sum(int(w) << (32 * i) for i, w in enumerate(r[1:]))) for r in got["checksums"]] == checksums
    rows = got["sample_rows"].astype(np.int64)
    assert rows.size == 100 and np.all(np.diff(rows) > 0) and rows[-1] < 1000
    assert np.array_equal(got["transform"], orc.read_component(cols[0], 0, 1000)[rows].view(np.float32))
    assert np.array_equal(got["ttl"], orc.read_component(cols[2], 0, 1000)[rows].view(np.uint64)[:, 0].astype(np.float64))
    orc.close()


def test_reference_arm_prints_the_contract_line_on_a_cpu_box():
    """`bench.py --impl reference` = the reference's CPU path (the oracle port here: no cargo, no checkout on the GPU box)
    on host cores, same metric / unit / config keys as our arm, bounded sample, no GPU needed."""
    import json
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "stress_100k_d8",
                        "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "rollback frames/s" and line["higher_is_better"] is True
    assert line["config"]["workload"] == "stress_100k_d8" and line["gpu_launches"] == 0
    assert line["cpu_baseline"]["kind"] in ("port", "reference") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "rollback frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["value"] > 0


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True,
                       text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""
