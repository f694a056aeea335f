"""GPU suite: bench.py --dump-outputs writes what the last timed step computed -- every frame's JPEG size and status and the
JPEG bytes of a sample of frames, as float arrays -- and those bytes are the encoder's real output for the bench's frames.
Four sub-batches on two slots, so that slots are reused inside the step whose output is kept."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_last_timed_step(orc, tmp_path):
    import torch

    import bench

    w, h, F = 322, 242, 64
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--frames", str(F), "--sub-batch", "16",
                        "--slots", "2", "--width", str(w), "--height", str(h), "--parity-frames", "2", "--sustain-seconds", "0", "--no-e2e",
                        "--no-cpu-baseline", "--no-overlap", "--no-extras", "--no-other-configs", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    arrays = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert set(arrays) == {"jpeg_sizes", "status", "sample_frames", "sample_jpeg_bytes"}
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= bench.DUMP_BYTES
    sizes, frames, data = arrays["jpeg_sizes"].astype(np.int64), arrays["sample_frames"].astype(np.int64), arrays["sample_jpeg_bytes"]
    assert len(sizes) == F and (sizes > 0).all() and (arrays["status"] == 0).all()
    assert frames.tolist() == bench.dump_sample(F) and len(data) == sizes[frames].sum()
    d_frames, fb, _ = bench.make_frames_torch(F, w, h, torch.device("cuda", 0))
    at = 0
    for i in frames:
        got = data[at: at + sizes[i]].astype(np.uint8).tobytes()
        at += sizes[i]
        assert got == bench.oracle_jpeg(d_frames[i, :fb].cpu().numpy(), w, h), f"frame {i}"
