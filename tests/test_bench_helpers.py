"""CPU suite: the parts of bench.py that do not need a GPU -- the JSON line goes to the saved stdout only, the NUMA binding
is a no-op when the topology cannot be read, the clock sampler degrades to "no samples" instead of failing, and the
reference arm prints the contract's keys."""
import io
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_numa_local_is_a_no_op_without_topology():
    import bench

    before = os.sched_getaffinity(0)
    n = bench.NumaLocal(0)
    with n:
        inside = os.sched_getaffinity(0)
    assert os.sched_getaffinity(0) == before
    assert n.node is not None or inside == before


def test_clock_sampler_degrades():
    import bench

    s = bench.ClockSampler(0)
    s.start()
    out = s.stop()
    assert set(out) >= {"sm_mhz", "sm_max_mhz", "reasons"}


def test_emit_line_is_one_json_line():
    import bench

    buf = io.StringIO()
    old = bench._json_out
    bench._json_out = buf
    try:
        bench.emit_line({"metric": bench.METRIC, "value": 1.0})
    finally:
        bench._json_out = old
    lines = buf.getvalue().splitlines()
    assert len(lines) == 1 and json.loads(lines[0])["value"] == 1.0


def test_reference_arm_line_has_the_contract_keys():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-frames", "4",
                        "--width", "320", "--height", "240"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-500:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_sample_indices_hold_first_last_and_stay_in_range():
    import bench

    for n, c in ((2048, 16), (64, 3), (2, 16), (1, 4)):
        pick = bench.sample_indices(n, c, seed=n)
        assert pick[0] == 0 and pick[-1] == n - 1 and len(pick) == min(max(c, len({0, n - 1})), n) and len(set(pick)) == len(pick)
        assert all(0 <= i < n for i in pick)


def test_dump_outputs_stay_within_budget_as_float_arrays(tmp_path):
    """The dump's frame sample is fixed by the arguments; the frames written are the sample's first ones that fit DUMP_BYTES,
    all of them when the JPEGs are small, none when not even one fits."""
    import numpy as np

    import bench

    F = 2048
    pick = bench.dump_sample(F)
    assert pick == bench.dump_sample(F) and pick[0] == 0 and pick[-1] == F - 1 and len(pick) == 16
    rng = np.random.default_rng(3)
    for size, n_written in ((300_000, 16), (2 * 1024 * 1024, 7), (17_000_000, 0)):
        last = {"sizes": np.full(F, size, np.int64), "status": np.zeros(F, np.int64),
                "jpeg": {i: rng.integers(0, 256, size, dtype=np.uint8) for i in pick}}
        out = tmp_path / str(size)
        bench.dump_outputs(str(out), last)
        files = sorted(os.listdir(out))
        assert files == ["jpeg_sizes.npy", "sample_frames.npy", "sample_jpeg_bytes.npy", "status.npy"]
        assert sum(os.path.getsize(out / f) for f in files) <= bench.DUMP_BYTES
        got = {f[:-4]: np.load(out / f) for f in files}
        assert all(a.dtype in (np.float32, np.float64) for a in got.values())
        assert got["sample_frames"].tolist() == pick[:n_written]
        assert (got["jpeg_sizes"] == size).all() and (got["status"] == 0).all()
        want = np.concatenate([np.zeros(0, np.uint8)] + [last["jpeg"][i] for i in pick[:n_written]])
        assert got["sample_jpeg_bytes"].shape == want.shape and (got["sample_jpeg_bytes"].astype(np.uint8) == want).all()


def test_device_plans(monkeypatch, tmp_path):
    import bench

    class FakeCuda:
        def __init__(self, n):
            self.n = n

        def device_count(self):
            return self.n

    class FakeTorch:
        def __init__(self, n):
            self.cuda = FakeCuda(n)

    # the measured rates of the pool's 8-GPU box: GPUs 4-7 are the good ones
    rates = [23.6, 23.6, 23.6, 23.6, 36.1, 36.2, 36.2, 36.1]
    assert bench.pick_devices(rates, 4) == [4, 5, 6, 7]
    assert bench.pick_devices(rates, 2) == [4, 5]
    assert bench.pick_devices([55.0] * 8, 4) == [0, 1, 2, 3]
    # as many ranks as GPUs, one rank, or the knob: identity
    assert bench.device_plan(FakeTorch(8), 0, 1)[0] == 0
    monkeypatch.setenv("H2J_BENCH_SPREAD", "0")
    assert [bench.device_plan(FakeTorch(8), r, 2)[0] for r in range(2)] == [0, 1]
    assert [bench.device_plan(FakeTorch(8), r, 8)[0] for r in range(8)] == list(range(8))
    monkeypatch.delenv("H2J_BENCH_SPREAD")
    # fewer ranks than GPUs, no usable probe here (no GPU): local rank 0 publishes the even spread, the others read it
    monkeypatch.setattr(bench.tempfile, "gettempdir", lambda: str(tmp_path))
    monkeypatch.setenv("MASTER_PORT", "29999")
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))  # no pcie_probe binary under this root
    assert bench.device_plan(FakeTorch(8), 0, 4)[0] == 0
    assert [bench.device_plan(FakeTorch(8), r, 4)[0] for r in range(1, 4)] == [2, 4, 6]
    assert bench.device_plan(FakeTorch(8), 3, 4)[2] is None  # no rates without a probe: equal shards
