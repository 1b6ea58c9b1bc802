"""Host-side logic of bench.py that needs no GPU: the two-node pipeline harness."""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def test_two_stage_pipeline_orders_and_gates():
    import bench
    log = []
    started = {}

    def stage_a(k, b):
        time.sleep(0.002)
        log.append(("a", k, b))
        return k * 10

    def stage_b(k, b, item):
        assert item == k * 10
        time.sleep(0.003)
        log.append(("b", k, b))

    def on_start():
        started["a_done"] = [x[1] for x in log if x[0] == "a"]
        started["b_done"] = [x[1] for x in log if x[0] == "b"]

    bench.run_two_stage_pipeline(12, 4, 3, stage_a, stage_b, on_start, lambda: log.append(("end",)), timeout_s=10.0)
    assert started["a_done"] == [0, 1, 2, 3] and started["b_done"] == [0, 1, 2, 3]      # warm-up fully drained before the clock starts
    assert [x[1] for x in log if x[0] == "b"] == list(range(12)) and log[-1] == ("end",)
    # never more than nbuf scans in flight
    inflight = 0
    for x in log:
        if x[0] == "a": inflight += 1
        elif x[0] == "b": inflight -= 1
        assert inflight <= 3
    bench.run_two_stage_pipeline(5, 0, 2, stage_a, stage_b, lambda: None, lambda: None, timeout_s=10.0)   # no warm-up


def test_two_stage_pipeline_propagates_errors():
    import bench
    import pytest

    def boom(k, b, item):
        raise ValueError("stage b failed")
    with pytest.raises(ValueError):
        bench.run_two_stage_pipeline(6, 2, 2, lambda k, b: k, boom, lambda: None, lambda: None, timeout_s=5.0)


def test_tools_and_entry_points_compile():
    """Every script a GPU session runs (tools/, bench.py, __graft_entry__.py, fixture generators) must at least parse."""
    import glob
    import py_compile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    files = glob.glob(os.path.join(root, "tools", "*.py")) + [os.path.join(root, f) for f in ("bench.py", "__graft_entry__.py")] + \
        glob.glob(os.path.join(root, "tests", "make_golden*.py"))
    assert len(files) >= 8
    for f in files:
        py_compile.compile(f, doraise=True)


def test_workload_resolution_and_shared_config():
    """Both bench arms (ours / --impl reference) must describe the SAME workload with the SAME `config` object, at N = 1 (configs[1])
    and at N > 1 (the streamed configs[4] workload, sharded)."""
    import argparse
    import bench
    a = argparse.Namespace(multi="sharded", workload="", map_points=0)
    assert bench.resolve_workload(a, 1) == ("horizon", 1_000_000)
    assert bench.resolve_workload(a, 8) == ("stream", 10_000_000)
    a.multi = "replicas"
    assert bench.resolve_workload(a, 8) == ("horizon", 1_000_000)
    a.workload = "rot"
    assert bench.resolve_workload(a, 1) == ("rot", 2_000_000)
    c1 = bench.config_dict("stream", 127788, 10_000_000, 8, "sharded")
    c2 = bench.config_dict("stream", 127788, 10_000_000, 8, "sharded")
    assert c1 == c2 and c1["map_frames"] == bench.N_FRAMES and "streamed" in c1["workload"] and c1["multi"] == "sharded"
    assert bench.config_dict("horizon", 20458, 1_000_000, 1, "sharded")["multi"] == "single"


def test_stream_frames_partition_the_map():
    """The streamed workload's 20 frames are a partition of the synthetic map (equal slabs along x, oldest first)."""
    import numpy as np
    import bench
    from liliom_b200 import synth
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__))))
    import oracle_lib as O
    m, _ = synth.make_map(50_000)
    frames = bench.make_frames(m, O.PT32)
    assert len(frames) == bench.N_FRAMES and sum(len(f) for f in frames) == len(m)
    allx = np.concatenate([f["x"] for f in frames])
    assert np.all(np.diff(allx) >= 0)                                   # slabs in ascending x
    got = np.sort(np.stack([np.concatenate([f[k] for f in frames]) for k in ("x", "y", "z")], 1).view([("", "f4")] * 3), axis=0)
    want = np.sort(np.ascontiguousarray(m[:, :3]).view([("", "f4")] * 3), axis=0)
    assert np.array_equal(got, want)


def test_clock_sampler_keeps_the_rows_inside_the_window(tmp_path, monkeypatch):
    """The clocks line of the bench comes from ONE looping `nvidia-smi -lms` process started before the timed region; only rows that
    arrive inside the window count.  Driven here by a stand-in nvidia-smi (no GPU in this container)."""
    import stat
    import time
    import bench
    fake = tmp_path / "nvidia-smi"
    fake.write_text("#!/bin/bash\n"
                    "# stand-in: the first rows report a low clock (before the window), later rows the full clock with a power cap\n"
                    "for i in $(seq 1 400); do\n"
                    "  if [ $i -le 8 ]; then echo '345, 1965, Not Active, Not Active, Not Active, Not Active';\n"
                    "  else echo '1965, 1965, Not Active, Not Active, Not Active, Active'; fi\n"
                    "  sleep 0.025\n"
                    "done\n")
    fake.chmod(fake.stat().st_mode | stat.S_IEXEC)
    monkeypatch.setenv("PATH", str(tmp_path) + os.pathsep + os.environ.get("PATH", ""))
    clk = bench.ClockSampler(0, enabled=True).start()
    time.sleep(0.5)                                  # "workload construction": rows from here must not count
    with clk:
        time.sleep(0.4)                              # the timed region
    s = clk.summary()
    assert s["samples"] >= 8 and s["sm_mhz"] == 1965.0 and s["sm_max_mhz"] == 1965.0
    assert s["reasons"] == ["sw_power_cap"] and s["period_ms"] == bench.ClockSampler.PERIOD_MS
    # disabled sampler (ranks != 0): no process, empty summary
    off = bench.ClockSampler(0, enabled=False).start()
    with off:
        pass
    assert off.summary()["samples"] == 0 and off.summary()["sm_mhz"] is None


def test_dump_outputs_types_and_budget(tmp_path, monkeypatch):
    """--dump-outputs: clouds become [n, fields] float32 with their bits kept, the pose stays float64, counts become float64;
    over the size budget every cloud keeps the same seeded sample of rows, identical from run to run, and the pose stays whole."""
    import numpy as np
    import bench
    from liliom_b200 import PT48
    cloud = np.zeros(1000, PT48)
    cloud["x"] = np.arange(1000, dtype=np.float32); cloud["curvature"] = 0.1
    pose = np.array([1.0, 0, 0, 0, 0.1, 0.2, 0.3])
    bench.dump_outputs(str(tmp_path / "a"), {"surf": cloud, "pose": pose, "queries": [1409]})
    s = np.load(tmp_path / "a" / "surf.npy")
    assert s.dtype == np.float32 and s.shape == (1000, 12) and s.tobytes() == cloud.tobytes()
    p = np.load(tmp_path / "a" / "pose.npy")
    assert p.dtype == np.float64 and p.tobytes() == pose.tobytes()
    assert np.load(tmp_path / "a" / "queries.npy").tolist() == [1409.0]
    monkeypatch.setattr(bench, "DUMP_BUDGET_BYTES", 12_000)
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), {"surf": cloud, "pose": pose})
    b, c = np.load(tmp_path / "b" / "surf.npy"), np.load(tmp_path / "c" / "surf.npy")
    assert sum(np.load(tmp_path / "b" / f).nbytes for f in ("surf.npy", "pose.npy")) <= 12_000
    assert 0 < len(b) < 1000 and np.array_equal(b, c) and np.all(np.diff(b[:, 0]) > 0)
    assert np.load(tmp_path / "b" / "pose.npy").tobytes() == pose.tobytes()


def test_two_node_leg_is_fail_safe():
    """bench.resolve_e2e: the optional two-node e2e leg may fail on any rank; then EVERY rank reports the one-thread figure (decided on
    the gathered per-rank times, so the ranks' collectives stay matched) and the line says so."""
    import bench
    seq = (123.0, ("pose", 1, 2))
    # one process, leg fine
    ms, last, err = bench.resolve_e2e(lambda: (40.0, ("p", 3, 4)), lambda m: (m, [m]), *seq)
    assert (ms, last, err) == (40.0, ("p", 3, 4), None)
    # one process, leg raises
    def boom():
        raise RuntimeError("exchange timed out")
    ms, last, err = bench.resolve_e2e(boom, lambda m: (m, [m]), *seq)
    assert ms == 123.0 and last == ("pose", 1, 2) and "RuntimeError: exchange timed out" in err
    # eight ranks, this one fine, another one failed: same fallback, and the gather was entered exactly once
    calls = []
    def gather(m):
        calls.append(m)
        return None, [m, 41.0, float("nan"), 39.0, 40.0, 40.0, 40.0, 40.0]
    ms, last, err = bench.resolve_e2e(lambda: (40.0, ("p", 3, 4)), gather, *seq)
    assert ms == 123.0 and last == ("pose", 1, 2) and "another rank" in err and calls == [40.0]
    # eight ranks, all fine: the maximum over ranks
    ms, last, err = bench.resolve_e2e(lambda: (40.0, ("p", 3, 4)), lambda m: (None, [m, 41.0, 39.5, 39.0, 40.0, 40.0, 40.0, 40.0]), *seq)
    assert ms == 41.0 and err is None and last == ("p", 3, 4)
