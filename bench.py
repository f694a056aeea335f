#!/usr/bin/env python
"""bench.py — JPEG encodes/s of the B200 YUV->JPEG path on synthetic textured 1080p frames.

  python bench.py --gpus N --steps K --warmup W            # our arm (N>1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's ffmpeg-mjpeg CPU path on the host cores
  python bench.py --steps K --dump-outputs DIR             # also writes what the last timed step computed, DIR/<name>.npy

A step is one pass of the hot path over one batch of `--frames` distinct frames (default 2048 x 1080p = 6.4 GB
of input, larger than the 126 MB L2, so nothing is served from cache between steps).
  value : frames/s, whole job, inputs already resident in HBM (h2j_submit_device), CUDA-event timed.
  e2e   : frames/s through the public C ABI with HOST buffers: pinned I420 frames in (H2D every step), JPEG
          bytes out to pinned host memory (D2H every step), wall-clock between device synchronisations.
  roofline : the dominant kernel's algorithmic bytes / its CUDA-event duration, against MEASURED_PEAKS.json.
  cpu_baseline : the compiled reference (oracle/_ref, the reference's own Encoder.cpp + vendored libavcodec)
          timed on this box's host cores on a bounded sample of the same frames.
Frames shard across ranks with no collective (images are independent): scaling is "weak".
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "h264-h265-to-jpeg_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "jpeg_encodes_per_sec_1080p"
UNIT = "frames/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--frames", type=int, default=2048, help="frames per step per GPU")
    ap.add_argument("--sub-batch", type=int, default=0, help="frames per submitted batch of the device-resident pass (0 = --frames)")
    ap.add_argument("--slots", type=int, default=1, help="batches in flight (streams) of the device-resident pass; 1 keeps the per-kernel "
                                                         "CUDA-event brackets free of other streams' kernels")
    ap.add_argument("--e2e-sub-batch", type=int, default=64, help="frames per submitted batch of the host-to-host pass")
    ap.add_argument("--e2e-slots", type=int, default=4, help="batches in flight of the host-to-host pass (overlaps H2D, kernels, D2H)")
    ap.add_argument("--cpu-frames", type=int, default=0, help="frames in the CPU baseline sample (0 = auto)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="wall time the CPU baseline sample should take")
    ap.add_argument("--max-jpeg-bytes", type=int, default=0, help="per-frame output capacity (0 = 2 MiB, the reference's HEAP_SIZE)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-every", type=int, default=5, help="per-kernel CUDA-event brackets on every K-th timed step (1 = all)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="skip the informational two-stream pass")
    ap.add_argument("--no-extras", action="store_true", help="skip the single-picture and IDecoder::H265ToJpeg records")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the 4K and 1918x1078 records (BASELINE.json configs[3])")
    ap.add_argument("--parity-frames", type=int, default=16, help="frames of the last timed launch compared with the oracle")
    ap.add_argument("--sustain-seconds", type=float, default=3.0, help="length of the sustained device-resident pass (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step of the device-resident "
                                                          "pass computed as DIR/<name>.npy (rank 0's frames; see dump_outputs).  The "
                                                          "frames are read after the timed region, except with more sub-batches than "
                                                          "slots: then a reused slot's are read inside it, which the timing includes")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs dumps the GPU path's outputs; the reference arm has none to write")
    return a


# ------------------------------------------------------------------------------------------------------
# synthetic workload: textured frames (smooth gradients + band-limited texture + mild noise), made on the GPU
# ------------------------------------------------------------------------------------------------------
def make_frames_torch(n, w, h, device, seed0=0, chroma_format=0):
    import torch

    import h2j_b200

    ch, cw = h2j_b200.chroma_shape(w, h, chroma_format)
    fb = w * h + 2 * cw * ch
    stride = (fb + 255) // 256 * 256
    out = torch.zeros((n, stride), dtype=torch.uint8, device=device)
    g = torch.Generator(device=device)

    def plane(hh, ww, amp, seed):
        yy = torch.arange(hh, device=device, dtype=torch.float32)[:, None]
        xx = torch.arange(ww, device=device, dtype=torch.float32)[None, :]
        s = float(seed % 97)
        p = 128 + 50 * torch.sin(xx / 97.0 + s) * torch.cos(yy / 61.0 - s) + amp * torch.sin(xx / 3.1 + yy / 4.3 + s) * torch.sin(yy / 2.3 + 0.37 * s)
        g.manual_seed(seed)
        p = p + torch.randn((hh, ww), device=device, generator=g) * (amp / 6.0)
        return p.clamp(0, 255).to(torch.uint8)

    for i in range(n):
        seed = seed0 + i
        amp = 20 + (seed * 7) % 40  # varies the rate-control outcome from frame to frame
        out[i, : w * h] = plane(h, w, amp, 3 * seed).reshape(-1)
        out[i, w * h: w * h + cw * ch] = plane(ch, cw, amp // 2, 3 * seed + 1).reshape(-1)
        out[i, w * h + cw * ch: fb] = plane(ch, cw, amp // 2, 3 * seed + 2).reshape(-1)
    return out, fb, stride


def make_frames_numpy(n, w, h, seed0=0):
    from tests.support import oracle as orc

    base = [orc.pack_i420(*orc.synth_planes(w, h, "textured", seed=seed0 + s, amp=20 + (s * 7) % 40)) for s in range(min(n, 8))]
    return np.stack([base[i % len(base)] for i in range(n)])


# ------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region.  NVML is polled from a thread every couple of milliseconds
    (the timed region of the default run lasts ~30 ms: `nvidia-smi -lms` does not even start up in that time, which is
    what an 8-GPU run showed); `nvidia-smi` stays as the fallback when the NVML binding is missing."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.h = None
        self.p = None
        self.f = None
        self.thread = None
        self.samples = []
        try:
            import pynvml
            import torch

            pynvml.nvmlInit()
            pr = torch.cuda.get_device_properties(gpu_index)
            bus = f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
            self.h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    def _poll(self):
        nv = self.nv
        while not self._stop:
            try:
                self.samples.append((float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)),
                                     int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))))
            except Exception:
                break
            time.sleep(0.002)

    def start(self):
        if self.h is not None:
            import threading

            self._stop = False
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.p = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.thread is not None:
            self._stop = True
            self.thread.join(timeout=2)
            if not self.samples:
                return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["no samples"], "source": "nvml"}
            nv = self.nv
            names = (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                     ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap),
                     ("hw_power_brake_slowdown", nv.nvmlClocksEventReasonHwPowerBrakeSlowdown))
            reasons = sorted({n for _, r in self.samples for n, bit in names if r & bit})
            return {"sm_mhz": float(np.median([m for m, _ in self.samples])), "sm_max_mhz": self.max_mhz, "reasons": reasons,
                    "samples": len(self.samples), "source": "nvml, polled every 2 ms during the timed region"}
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].strip().lower() == "active":
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 100"}


# ------------------------------------------------------------------------------------------------------
# host memory placement: pinned buffers are allocated (and first touched) on the GPU's own NUMA node
# ------------------------------------------------------------------------------------------------------
class NumaLocal:
    """Context manager: while active, the process runs on the CPUs of the NUMA node the GPU hangs off, so that the
    page-locked buffers allocated inside land in that node's memory (one PCIe root away from the GPU instead of across
    the socket interconnect -- matters when eight ranks pull 50 GB/s each).  The previous affinity is restored on exit:
    the CPU baseline and everything else keep all the cores.  Does nothing when the topology cannot be read."""

    def __init__(self, device_index):
        self.node = None
        self.saved = None
        try:
            import torch

            pr = torch.cuda.get_device_properties(device_index)
            bus = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
            node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
            if node < 0:
                return
            cpus = set()
            for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
            self.cpus = cpus & os.sched_getaffinity(0)
            if self.cpus:
                self.node = node
        except Exception:
            self.node = None

    def __enter__(self):
        if self.node is not None:
            self.saved = os.sched_getaffinity(0)
            os.sched_setaffinity(0, self.cpus)
        return self

    def __exit__(self, *exc):
        if self.saved is not None:
            os.sched_setaffinity(0, self.saved)
        return False

# ------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline
# ------------------------------------------------------------------------------------------------------
def reference_lib():
    from tests.support import oracle as orc

    if not orc.have_reference():
        return None
    lib = orc.reference()
    lib.ref_yuv2jpeg_batch_mt.argtypes = [C.c_void_p, C.c_long, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
    return lib


def cpu_encode_sample(frames: np.ndarray, w, h, n, threads):
    """Encode n frames (cycling over `frames`) on `threads` host threads; returns (seconds, kind)."""
    from tests.support import oracle as orc

    reps = (n + frames.shape[0] - 1) // frames.shape[0]
    sample = np.ascontiguousarray(np.concatenate([frames] * reps)[:n])
    sizes = np.zeros(n, np.int64)
    ref = reference_lib()
    if ref is not None:
        t0 = time.perf_counter()
        ok = ref.ref_yuv2jpeg_batch_mt(sample.ctypes.data, sample.shape[1], n, w, h, sizes.ctypes.data, threads)
        dt = time.perf_counter() - t0
        assert ok == n, f"reference encoded {ok}/{n} frames"
        return dt, "reference", sizes
    lib = orc.oracle()
    p = orc.Params(w, h, orc.NOPTS, 0, 0, None)
    cap = 4 * 1024 * 1024
    out = np.empty(cap * min(n, 64), np.uint8)
    t0 = time.perf_counter()
    done = 0
    while done < n:
        m = min(64, n - done)
        lib.orc_encode_batch_mt(sample[done:].ctypes.data, sample.shape[1], m, C.byref(p), out.ctypes.data, cap, sizes[done:].ctypes.data, threads)
        done += m
    return time.perf_counter() - t0, "port", sizes


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    w, h = a.width, a.height
    cores = os.cpu_count() or 1
    frames = make_frames_numpy(8, w, h)
    # bounded sample per step: sized from a calibration pass so that warmup + steps take about a minute in all
    n0 = max(2 * cores, 16)
    dt0, _, _ = cpu_encode_sample(frames, w, h, n0, cores)
    per_step_s = min(6.0, 60.0 / max(1, a.steps + a.warmup))
    n = a.cpu_frames or max(n0, int(per_step_s * n0 / dt0))
    for _ in range(a.warmup):
        cpu_encode_sample(frames, w, h, n, cores)
    times = []
    kind = "port"
    for _ in range(a.steps):
        dt, kind, _ = cpu_encode_sample(frames, w, h, n, cores)
        times.append(dt)
    total = sum(times)
    value = n * a.steps / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1000 * total / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/int16",
        "data": "synthetic", "mpixel_per_s": value * w * h / 1e6,
        "config": {"workload": f"{n} synthetic textured {w}x{h} yuv420p frames per step through the reference's Encoder::yuv2Jpeg "
                               f"(ffmpeg mjpeg, libavcodec 58.117.101) on {cores} host threads; stock path: every frame is copied into a fresh "
                               "AVFrame and its JPEG written to a tmpfs file by the reference's own saveJpegtoFile",
                   "host_cores": cores},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": f"{n} frames x {a.steps} steps"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_line(line)


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
class Ctx:
    """What every pass of a rank needs: device, ranks, barrier and max-over-ranks."""

    def __init__(self, torch, dist, dev, rank, world):
        self.torch, self.dist, self.dev, self.rank, self.world = torch, dist, dev, rank, world

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x, dtype=None):
        t = self.torch.tensor([x], device=self.dev, dtype=dtype or self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather(self, x):
        """x of every rank, as a list (rank order)."""
        g = self.torch.zeros(self.world, device=self.dev, dtype=self.torch.float64)
        g[self.rank] = x
        if self.world > 1:
            self.dist.all_reduce(g, op=self.dist.ReduceOp.SUM)
        return [float(v) for v in g.tolist()]


def pick_devices(per_gpu_gbs, world):
    """The `world` GPUs with the best host->device rate when every GPU of the box copies at once (ties: lower ordinal),
    in ascending order."""
    order = sorted(range(len(per_gpu_gbs)), key=lambda g: (-round(per_gpu_gbs[g], 0), g))
    return sorted(order[:world])


def device_plan(torch, local_rank, world):
    """GPU of a rank, and every rank's host->device rate.  The host-to-host pass is bound by the host->device link, and
    on the 8-GPU boxes of this pool the GPUs are not equal there: GPUs 0-3 share ~117 GB/s of host reads, GPUs 4-7 get 55
    GB/s each, all eight together 24 + 36 GB/s (profiles/r2g_pcie_probe.jsonl), while `nvidia-smi topo -m` shows one flat
    NUMA node (the VM hides the sockets).  So a multi-rank job asks the box: local rank 0 runs tools/microbench/pcie_probe
    (plain pinned cudaMemcpyAsync on all GPUs at once, in a process of its own), a job with fewer ranks than visible GPUs
    takes the GPUs with the best rates, and the host-to-host pass sizes the ranks' shards by their rates
    (h2j_b200.weighted_shards).  H2J_BENCH_SPREAD=0 keeps rank i on GPU i with equal shards; if the probe is not there the
    ranks are spread evenly over the ordinals.  Returns (device ordinal, description, rates of the ranks' GPUs or None)."""
    n = torch.cuda.device_count()
    if world <= 1 or n < world or os.environ.get("H2J_BENCH_SPREAD", "1") == "0":
        return local_rank, f"identity: rank i on GPU i of {n} visible", None
    share = os.path.join(tempfile.gettempdir(), f"h2j_bench_devices_{os.getppid()}_{os.environ.get('MASTER_PORT', '0')}.json")
    if local_rank == 0:
        plan, why = None, "unusable output"
        try:
            exe = os.path.join(ROOT, "tools", "microbench", "pcie_probe")
            r = subprocess.run([exe, "all"], capture_output=True, text=True, timeout=120)
            rates = json.loads(r.stdout.strip().splitlines()[-1])["h2d_gbs_per_gpu"]
            if len(rates) == n and min(rates) > 0:
                gpus = pick_devices(rates, world)
                plan = {"gpus": gpus, "rates": [rates[g] for g in gpus], "how": f"probe: H2D GB/s per GPU with all {n} copying at once = {rates}"}
        except Exception as ex:
            why = str(ex)[:80]
        if plan is None:
            step = n // world
            plan = {"gpus": [i * step for i in range(world)], "rates": None, "how": f"no probe ({why}): every {step}-th GPU of {n}"}
        with open(share + ".tmp", "w") as f:
            json.dump(plan, f)
        os.replace(share + ".tmp", share)
    t0 = time.time()
    while not os.path.exists(share):
        if time.time() - t0 > 180:
            return local_rank, "identity: the device plan of local rank 0 never arrived", None
        time.sleep(0.05)
    plan = json.load(open(share))
    return plan["gpus"][local_rank], f"rank i on GPU {plan['gpus']}[i] -- {plan['how']}", plan["rates"]


def oracle_jpeg(frame_bytes, w, h, chroma_format=0):
    """JPEG the oracle (CPU restatement of the reference's encoder) makes of one tight planar frame."""
    import h2j_b200
    from tests.support import oracle as orc

    y, u, v = h2j_b200.split_planes(frame_bytes, w, h, chroma_format)
    return orc.oracle_encode(np.ascontiguousarray(y), np.ascontiguousarray(u), np.ascontiguousarray(v), chroma_format=chroma_format)[0]


def sample_indices(n, count, seed):
    """first, last and random frames of a batch of n"""
    rng = np.random.default_rng(seed)
    pick = {0, n - 1}
    while len(pick) < min(count, n):
        pick.add(int(rng.integers(0, n)))
    return sorted(pick)


def device_pass(cx, enc, streams, d_frames, stride, fb, F, SB, NS, w, h, steps, warmup, profile_every, sample=0, min_seconds=0.0, chroma_format=0,
                keep_frames=()):
    """The device-resident pass: `steps` steps of F frames in sub-batches of SB on NS slots, CUDA-event timed.  After
    the timed region `sample` frames of the LAST timed launch are fetched from the device and compared with the oracle.
    min_seconds > 0: keep stepping until the timed region has lasted that long (sustained figure).
    keep_frames: frames (indices within a step) whose JPEG bytes the last timed step keeps; out["last_step"] then holds
    them and the sizes and status of every frame of that step.  They are read after the timed region, except from a slot
    that the step reuses (more sub-batches than slots): that slot's are read before its next submit, inside the region."""
    torch = cx.torch
    nsub = F // SB
    main = torch.cuda.current_stream(cx.dev)
    kernel_ms, kernel_calls = {}, {}
    sizes_total = [0]
    last = {}
    kept = {"sizes": np.zeros(F, np.int64), "status": np.zeros(F, np.int64), "jpeg": {}, "launches": []}

    def harvest(slot):
        for name, ms in enc.kernel_ms(slot):
            kernel_ms[name] = kernel_ms.get(name, 0.0) + ms
            kernel_calls[name] = kernel_calls.get(name, 0) + 1

    def collect(slot, first_frame, record, keep):
        d_out, cap, sizes, st = enc.collect_device(slot)
        if record:
            harvest(slot)
            sizes_total[0] += int(sizes.sum())
            last.update(slot=slot, first_frame=first_frame, d_out=d_out, cap=cap, sizes=sizes, status=st)
        if keep:
            kept["sizes"][first_frame: first_frame + len(sizes)] = sizes
            kept["status"][first_frame: first_frame + len(st)] = st
            kept["launches"].append((first_frame, d_out, cap, sizes))

    def read_kept():
        for first_frame, d_out, cap, sizes in kept["launches"]:
            for i in keep_frames:
                j = i - first_frame
                if 0 <= j < len(sizes):
                    kept["jpeg"][i] = np.frombuffer(enc.read_device(d_out + j * cap, int(sizes[j])), np.uint8)
        kept["launches"].clear()

    def step(record=False, keep=False):
        inflight = []
        for i in range(nsub):
            slot = i % NS
            if len(inflight) == NS:
                s0, f0 = inflight.pop(0)
                collect(s0, f0, record, keep)
                if keep:
                    read_kept()
            enc.submit_device(slot, d_frames.data_ptr() + i * SB * stride, stride, SB, w, h)
            inflight.append((slot, i * SB))
        for s0, f0 in inflight:
            collect(s0, f0, record, keep)

    for _ in range(warmup):
        step()
    sampler = ClockSampler(cx.dev.index)
    cx.barrier()
    sampler.start()
    launches0 = enc.kernel_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(main)
    for st in streams:
        st.wait_stream(main)
    t0 = time.perf_counter()
    done = 0
    while done < steps or (min_seconds > 0 and time.perf_counter() - t0 < min_seconds):
        # per-kernel event brackets on a sample of the timed steps: a bracket leaves the GPU idle for a few microseconds at
        # every kernel boundary (eight per step), which is instrumentation, not the encoder
        enc.set_profile(profile_every > 0 and done % max(1, profile_every) == 0)
        step(record=True, keep=bool(keep_frames) and done == steps - 1 and min_seconds <= 0)
        done += 1
    for st in streams:
        main.wait_stream(st)
    ev1.record(main)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    cx.barrier()
    clocks = sampler.stop()
    dev_ms = ev0.elapsed_time(ev1)
    out = {"dev_ms": dev_ms, "dev_ms_max": cx.max_over_ranks(dev_ms), "steps": done, "wall_s": wall, "clocks": clocks,
           "launches": enc.kernel_launches - launches0, "kernel_ms": kernel_ms, "kernel_calls": kernel_calls,
           "avg_jpeg": sizes_total[0] / max(1, F * done), "parity": None}
    out["value"] = cx.world * F * done / (out["dev_ms_max"] / 1000.0)
    if keep_frames:
        read_kept()
        out["last_step"] = {"sizes": kept["sizes"], "status": kept["status"], "jpeg": kept["jpeg"]}
    if sample > 0 and last:
        # frames of the launch that was just timed (the slot's output stays valid until the next submit)
        try:
            n_last = len(last["sizes"])
            pick = sample_indices(n_last, sample, seed=F + w)
            bad = []
            for i in pick:
                got = enc.read_device(last["d_out"] + i * last["cap"], int(last["sizes"][i]))
                want = oracle_jpeg(d_frames[last["first_frame"] + i, :fb].cpu().numpy(), w, h, chroma_format)
                if got != want or int(last["status"][i]) != 0:
                    bad.append(last["first_frame"] + i)
            out["parity"] = {"frames": len(pick), "ok": not bad, "launch_frames": n_last, "differing": bad,
                             "what": f"JPEG bytes of {len(pick)} frames (first, last, random) of the last timed {n_last}-frame launch vs the oracle"}
        except Exception as ex:  # the bench still reports; the tests are the gate
            out["parity"] = {"frames": 0, "ok": False, "error": str(ex)}
    return out


def e2e_pass(cx, d_frames, stride, fb, F, ESB, ENS, w, h, steps, warmup, max_jpeg_bytes=0, sample=0, job_frames=None):
    """Host-to-host through the C ABI: pinned I420 frames in (H2D every step), packed JPEG bytes out to pinned host
    memory (D2H every step); wall clock between device synchronisations, max over ranks.  After the timed region one more
    (untimed) step runs with `sample` frames of its first, middle and last sub-batch compared with the oracle."""
    import h2j_b200

    torch = cx.torch
    ensub = F // ESB
    cap = max_jpeg_bytes or 2 * 1024 * 1024
    out_cap = ESB * ((cap + 15) // 16 * 16)
    numa = NumaLocal(cx.dev.index)
    with numa:
        enc = h2j_b200.Encoder(max_width=w, max_height=h, max_batch=ESB, n_slots=ENS, device=cx.dev.index, max_jpeg_bytes=max_jpeg_bytes)
        h_in = h2j_b200.PinnedBuffer(F * stride)
        h_in.array[:] = d_frames.reshape(-1).cpu().numpy()
        h_out = [h2j_b200.PinnedBuffer(out_cap) for _ in range(ENS)]
        for b in h_out:
            b.array[::4096] = 0
    d2h = [0]
    launches0 = enc.kernel_launches
    checks = {}

    def collect(slot, sub, check):
        offs, st = enc.collect_into(slot, h_out[slot].ptr, out_cap)
        d2h[0] += int(offs[-1])
        if check is not None and sub in check:
            for i in check[sub]:
                got = h_out[slot].array[int(offs[i]): int(offs[i + 1])].tobytes()
                checks[sub * ESB + i] = (got == oracle_jpeg(h_in.array[(sub * ESB + i) * stride: (sub * ESB + i) * stride + fb], w, h)) and int(st[i]) == 0

    def step(check=None):
        inflight = []
        for i in range(ensub):
            slot = i % ENS
            if len(inflight) == ENS:
                s0, sub0 = inflight.pop(0)
                collect(s0, sub0, check)
            enc.submit_host(slot, h_in.ptr + i * ESB * stride, stride, ESB, w, h)
            inflight.append((slot, i))
        for s0, sub0 in inflight:
            collect(s0, sub0, check)

    for _ in range(warmup):
        step()
    cx.barrier()
    d2h[0] = 0
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    cx.barrier()
    dt_max = cx.max_over_ranks(dt)
    per_rank_s = cx.gather(dt)
    job = job_frames if job_frames is not None else cx.world * F  # frames all ranks encode per step (F is THIS rank's share)
    res = {"value": job * steps / dt_max, "unit": UNIT, "h2d_bytes_per_step": job * fb,
           "d2h_bytes_per_step": int(sum(cx.gather(float(d2h[0])))) // max(1, steps), "timing": "wall clock between device synchronisations, max over ranks",
           "sub_batch": ESB, "slots": ENS, "h2d_gbs": job * fb * steps / dt_max / 1e9, "pinned_numa_node": numa.node,
           "per_rank": {"ms_per_step": [round(1000 * x / steps, 3) for x in per_rank_s],
                        "frames_per_step": [int(x) for x in cx.gather(float(F))],
                        "h2d_gbs": [round(f_ * fb * steps / x / 1e9, 2) for f_, x in zip(cx.gather(float(F)), per_rank_s)],
                        "gpu": cx.gather(float(cx.dev.index))},
           "gpu_launches": enc.kernel_launches - launches0,
           "note": "host-pinned I420 in, packed JPEG bytes out to pinned host memory, every step; bound by the H2D copy "
                   f"({fb / 1e6:.2f} MB of pixels per frame over PCIe)"}
    if sample > 0:
        try:
            subs = sorted({0, ensub // 2, ensub - 1})
            per = max(1, sample // len(subs))
            check = {sb: sample_indices(ESB, per, seed=sb + 1) for sb in subs}
            step(check)
            res["parity_sampled"] = {"frames": len(checks), "ok": all(checks.values()), "differing": [k for k, ok in checks.items() if not ok],
                                     "what": "JPEG bytes in the pinned output buffer vs the oracle, frames of the first, middle and last sub-batch of one more (untimed) step"}
        except Exception as ex:
            res["parity_sampled"] = {"frames": 0, "ok": False, "error": str(ex)}
    enc.close()
    h_in.free()
    for b in h_out:
        b.free()
    return res


def kernel_table(dp, w, h, fb, SB, peak, nblk=None):
    """Per-kernel averages and the algorithmic-bytes rates of DESIGN.md section 4."""
    mcu = ((w + 15) // 16) * ((h + 15) // 16)
    nblk = nblk or mcu * 6
    alg_bytes = algorithmic_bytes(w, h, fb, nblk, dp["avg_jpeg"], dp.get("avg_image_bytes"))
    per_kernel = {}
    for name, ms in dp["kernel_ms"].items():
        calls = dp["kernel_calls"][name]
        avg_ms = ms / calls
        entry = {"avg_ms": avg_ms, "launches": calls}
        if name in alg_bytes:
            entry["gbs"] = alg_bytes[name] * SB / (avg_ms * 1e-3) / 1e9
            entry["frac_of_hbm_peak"] = entry["gbs"] / peak
        per_kernel[name] = entry
    return per_kernel, alg_bytes


def algorithmic_bytes(w, h, fb, nblk, avg_jpeg, avg_image_bytes=None):
    """Bytes each kernel has to move per frame (DESIGN.md section 4)."""
    coef = avg_image_bytes if avg_image_bytes else nblk * 136
    return {
        "mbvar_kernel": w * h,
        "fdct_quant_kernel": fb + coef,
        "entropy_walk_kernel": coef + avg_jpeg,
        "scan_place_kernel": 2 * avg_jpeg,
        "stuff_kernel": 2 * avg_jpeg,
        "huffman_kernel": nblk * 2,
    }


DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this much


def dump_sample(F):
    """Frames of a step whose JPEG bytes --dump-outputs keeps: the first, the last and seeded random ones, 16 in all."""
    return sample_indices(F, 16, seed=F)


def dump_outputs(path, last):
    """What the last timed step handed its caller, as path/<name>.npy:
      jpeg_sizes         float64 [F]  bytes of every frame's JPEG
      status             float64 [F]  every frame's status (0 = ok)
      sample_frames      float64 [S]  the kept frames (dump_sample), in order, as many as fit DUMP_BYTES in all
      sample_jpeg_bytes  float32      the JPEG bytes of those frames, concatenated in frame order"""
    os.makedirs(path, exist_ok=True)
    room = (DUMP_BYTES - 16 * len(last["sizes"]) - 4 * 4096) // 4  # float32 bytes left after the per-frame arrays and npy headers
    frames = []
    for i in sorted(last["jpeg"]):
        room -= len(last["jpeg"][i]) + 2  # + 2: the frame's entry in sample_frames
        if room < 0:
            break
        frames.append(i)
    arrays = {"jpeg_sizes": last["sizes"].astype(np.float64), "status": last["status"].astype(np.float64),
              "sample_frames": np.array(frames, np.float64),
              "sample_jpeg_bytes": np.concatenate([np.zeros(0, np.uint8)] + [last["jpeg"][i] for i in frames]).astype(np.float32)}
    for name, arr in arrays.items():
        np.save(os.path.join(path, name + ".npy"), arr)


def hbm_peak():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    return peak, ("MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)")


def other_config(cx, w, h, F, ESB, a, chroma_format=0):
    """One of BASELINE.json configs[3]'s geometries (or, with chroma_format, the encoder's other MCU geometries), outside
    the headline: device-resident and host-to-host throughput, the FDCT kernel's roofline fraction and a parity sample of
    the timed launch."""
    import h2j_b200

    torch = cx.torch
    cap = 4 * 1024 * 1024 if w * h > 1920 * 1088 or chroma_format else 0
    d_frames, fb, stride = make_frames_torch(F, w, h, cx.dev, seed0=1000 + cx.rank * F, chroma_format=chroma_format)
    torch.cuda.synchronize()
    enc = h2j_b200.Encoder(max_width=w, max_height=h, max_batch=F, n_slots=1, device=cx.dev.index, profile=True, max_jpeg_bytes=cap, chroma_format=chroma_format)
    st = torch.cuda.Stream(device=cx.dev)
    enc.set_stream(0, st.cuda_stream)
    dp = device_pass(cx, enc, [st], d_frames, stride, fb, F, F, 1, w, h, steps=max(3, a.steps // 2), warmup=3, profile_every=2, sample=6, chroma_format=chroma_format)
    peak, _ = hbm_peak()
    nblk_fmt = ((w + 7) // 8) * ((h + 15) // 16) * 6 if chroma_format == 2 else ((w + 15) // 16) * ((h + 15) // 16) * (8 if chroma_format == 1 else 6)
    per_kernel, _ = kernel_table(dp, w, h, fb, F, peak, nblk=nblk_fmt)
    enc.close()
    rec = {"chroma_format": {0: "4:2:0", 1: "4:2:2", 2: "4:4:4"}[chroma_format], "width": w, "height": h, "frames_per_step_per_gpu": F, "value": dp["value"], "unit": UNIT, "mpixel_per_s": dp["value"] * w * h / 1e6,
           "ms_per_step": dp["dev_ms_max"] / dp["steps"], "steps": dp["steps"], "avg_jpeg_bytes": dp["avg_jpeg"], "parity_sampled": dp["parity"],
           "fdct_quant_kernel_frac": per_kernel.get("fdct_quant_kernel", {}).get("frac_of_hbm_peak"),
           "kernels_ms": {k: round(v["avg_ms"], 4) for k, v in per_kernel.items()}}
    if not a.no_e2e and chroma_format == 0:
        e2e = e2e_pass(cx, d_frames, stride, fb, F, ESB, 4, w, h, steps=max(2, a.steps // 3), warmup=2, max_jpeg_bytes=cap, sample=3)
        rec["e2e"] = {k: e2e[k] for k in ("value", "unit", "h2d_gbs", "sub_batch", "slots", "parity_sampled") if k in e2e}
    del d_frames
    torch.cuda.empty_cache()
    return rec


def camera_record(cx, F, a):
    """The encoder on the reference's OWN picture: test/img/img01.h264 (a 1920x1080 camera frame), decoded once on the host by
    the libavcodec the reference vendors (oracle/_ref), F copies of it device-resident.  The bench frames are synthetic texture
    with ~2.6 x the non-zero levels of this picture; this record says what the same kernels do on camera content.  Six frames
    of the timed launch are compared with the oracle."""
    import h2j_b200
    from tests.support import oracle as orc

    fix = os.path.join(ROOT, "oracle", "_ref", "fixtures", "img01.h264")
    if not orc.have_reference() or not os.path.exists(fix):
        return {"unavailable": "the compiled reference (its decoder) or the reference's test picture is not present on this box"}
    torch = cx.torch
    R = orc.reference()
    yb = np.zeros(4096 * 4096, np.uint8); ub = np.zeros(2048 * 2048, np.uint8); vb = np.zeros_like(ub)
    info = np.zeros(8, np.int64)
    if R.ref_decode_first_frame(fix.encode(), yb.ctypes.data, ub.ctypes.data, vb.ctypes.data, yb.size, info.ctypes.data) != 1:
        return {"error": "the reference's decoder did not return a frame"}
    w, h = int(info[0]), int(info[1])
    cw, ch = (w + 1) // 2, (h + 1) // 2
    frame = np.concatenate([yb[: w * h], ub[: cw * ch], vb[: cw * ch]])
    fb = frame.size
    stride = (fb + 255) // 256 * 256
    d_frames = torch.zeros((F, stride), dtype=torch.uint8, device=cx.dev)
    d_frames[:, :fb] = torch.from_numpy(frame).to(cx.dev)[None, :]
    torch.cuda.synchronize()
    enc = h2j_b200.Encoder(max_width=w, max_height=h, max_batch=F, n_slots=1, device=cx.dev.index, profile=True)
    st = torch.cuda.Stream(device=cx.dev)
    enc.set_stream(0, st.cuda_stream)
    dp = device_pass(cx, enc, [st], d_frames, stride, fb, F, F, 1, w, h, steps=max(3, a.steps // 2), warmup=3, profile_every=2, sample=6)
    peak, _ = hbm_peak()
    per_kernel, _ = kernel_table(dp, w, h, fb, F, peak)
    enc.close()
    del d_frames
    torch.cuda.empty_cache()
    return {"what": f"{F} copies of the reference's test picture img01.h264 ({w}x{h}, decoded by the reference's libavcodec), device-resident",
            "width": w, "height": h, "frames_per_step_per_gpu": F, "value": dp["value"], "unit": UNIT, "ms_per_step": dp["dev_ms_max"] / dp["steps"],
            "avg_jpeg_bytes": dp["avg_jpeg"], "parity_sampled": dp["parity"],
            "fdct_quant_kernel_frac": per_kernel.get("fdct_quant_kernel", {}).get("frac_of_hbm_peak"),
            "kernels_ms": {k: round(v["avg_ms"], 4) for k, v in per_kernel.items()}}


def nv12_record(cx, w, h, F, a):
    """Row f2 in the driver-run line: NV12 frames as a hardware decoder leaves them in HBM (luma and interleaved Cb/Cr
    planes at a 256-byte aligned pitch, the chroma plane behind the luma rows rounded up to 16), read in place by
    h2j_submit_device_nv12; device-resident throughput and frames of the timed launch against the oracle's JPEG of the
    equivalent planar frame."""
    import h2j_b200

    torch = cx.torch
    d_frames, fb, stride = make_frames_torch(F, w, h, cx.dev, seed0=3000 + cx.rank * F)
    cw, ch = (w + 1) // 2, (h + 1) // 2
    pitch = (max(w, 2 * cw) + 255) // 256 * 256
    uv_off = pitch * ((h + 15) // 16 * 16)
    nstride = (uv_off + pitch * ch + 255) // 256 * 256
    nv = torch.zeros((F, nstride), dtype=torch.uint8, device=cx.dev)
    nv[:, : pitch * h].view(F, h, pitch)[:, :, :w] = d_frames[:, : w * h].view(F, h, w)
    uv = nv[:, uv_off: uv_off + pitch * ch].view(F, ch, pitch)
    uv[:, :, 0: 2 * cw: 2] = d_frames[:, w * h: w * h + cw * ch].view(F, ch, cw)
    uv[:, :, 1: 2 * cw: 2] = d_frames[:, w * h + cw * ch: fb].view(F, ch, cw)
    torch.cuda.synchronize()
    enc = h2j_b200.Encoder(max_width=w, max_height=h, max_batch=F, n_slots=1, device=cx.dev.index)
    st = torch.cuda.Stream(device=cx.dev)
    enc.set_stream(0, st.cuda_stream)
    main = torch.cuda.current_stream(cx.dev)
    steps = max(3, a.steps // 2)

    def step():
        enc.submit_device_nv12(0, nv.data_ptr(), nstride, pitch, uv_off, F, w, h)
        return enc.collect_device(0)

    for _ in range(3):
        step()
    cx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(main)
    st.wait_stream(main)
    for _ in range(steps):
        d_out, cap, sizes, status = step()
    main.wait_stream(st)
    e1.record(main)
    torch.cuda.synchronize()
    cx.barrier()
    ms = cx.max_over_ranks(e0.elapsed_time(e1))
    bad = []
    pick = sample_indices(F, 6, seed=F + 12)
    for i in pick:
        got = enc.read_device(d_out + i * cap, int(sizes[i]))
        if got != oracle_jpeg(d_frames[i, :fb].cpu().numpy(), w, h) or int(status[i]) != 0:
            bad.append(i)
    enc.close()
    del nv, d_frames
    torch.cuda.empty_cache()
    return {"input": f"NV12 in HBM, read in place (pitch {pitch}, chroma plane at row {uv_off // pitch})", "width": w, "height": h, "frames_per_step_per_gpu": F,
            "value": cx.world * F * steps / (ms / 1000.0), "unit": UNIT, "steps": steps,
            "parity_sampled": {"frames": len(pick), "ok": not bad, "differing": bad,
                               "what": "JPEG bytes of frames of the last timed launch vs the oracle's JPEG of the planar frame with the same samples"}}


def single_frame_record(cx, w, h, d_frames, stride, fb):
    """The reference's own call shape (Encoder::yuv2Jpeg, one picture): host planes in, JPEG bytes out, synchronous."""
    import h2j_b200

    frame = d_frames[0, :fb].cpu().numpy()
    y, u, v = (np.ascontiguousarray(p) for p in h2j_b200.split_planes(frame, w, h))
    with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=1, n_slots=1, device=cx.dev.index) as e:
        for _ in range(20):
            got = e.yuv2jpeg(y, u, v)
        ts = []
        for _ in range(200):
            t0 = time.perf_counter()
            e.yuv2jpeg_into(y, u, v)
            ts.append(time.perf_counter() - t0)
        # the same call with the planes in page-locked memory (a decoder whose frame pool is pinned): no staging copy
        pin = h2j_b200.PinnedBuffer(fb)
        pin.array[:] = frame
        py, pu, pv = h2j_b200.split_planes(pin.array, w, h)
        tp = []
        for _ in range(20):
            e.yuv2jpeg_into(py, pu, pv)
        for _ in range(200):
            t0 = time.perf_counter()
            e.yuv2jpeg_into(py, pu, pv)
            tp.append(time.perf_counter() - t0)
        tp.sort()
        del py, pu, pv
        pin.free()
        # batch of one, device resident
        cx.torch.cuda.synchronize()
        for _ in range(20):
            e.submit_device(0, d_frames.data_ptr(), stride, 1, w, h)
            e.collect_device(0)
        t0 = time.perf_counter()
        for _ in range(300):
            e.submit_device(0, d_frames.data_ptr(), stride, 1, w, h)
            e.collect_device(0)
        dt = (time.perf_counter() - t0) / 300
    ts.sort()
    return {"what": f"h2j_encode_frame: one {w}x{h} picture, pageable host planes in, JPEG bytes out, synchronous (the Encoder::yuv2Jpeg call shape)",
            "ms_median": 1000 * ts[len(ts) // 2], "ms_p10": 1000 * ts[len(ts) // 10], "ms_p90": 1000 * ts[len(ts) * 9 // 10],
            "ms_median_pinned_planes": 1000 * tp[len(tp) // 2],
            "batch1_device_resident_fps": 1.0 / dt, "parity_ok": got == oracle_jpeg(frame, w, h)}


def dropin_record(cores):
    """configs[0]: the reference's real public call -- IDecoder::getInstance()->H265ToJpeg(in, out) on its own test pictures
    (the loop of the reference's main.cpp:37-65) -- through the drop-in library (the reference's Decoder.cpp + JNI bridge over
    this repo's Encoder) and through the unmodified reference, timed side by side on this box."""
    from tests.support import oracle as orc

    so = os.path.join(PKG, "lib", "libH265ToJpeg_b200.so")
    fix = os.path.join(ROOT, "oracle", "_ref", "fixtures")
    if not os.path.exists(so) or not os.path.isdir(fix):
        return {"unavailable": "drop-in library or the reference's test pictures not present on this box"}
    lib = C.CDLL(so)
    lib.dropin_loop.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]
    ref = None
    if orc.have_reference():
        ref = orc.reference()
        ref.ref_h265_loop.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]
    out = {"what": "IDecoder::H265ToJpeg(file in, JPEG file out): libavcodec decode of the picture + YUV->JPEG; outputs on tmpfs; "
                   "LOG() lines sent to /dev/null in both arms", "host_cores": cores, "pictures": {}}
    tmp = tempfile.mkdtemp(prefix="h2j_dropin_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        for name in ("img01.h265", "img01.h264"):
            src = os.path.join(fix, name).encode()
            rec = {}

            def ours(n, threads, batch, tag):
                sec = C.c_double()
                done = lib.dropin_loop(src, os.path.join(tmp, f"o_{tag}_").encode(), n, threads, batch, 1, C.byref(sec))
                return done, sec.value

            def theirs(n, threads, tag):
                sec = C.c_double()
                done = ref.ref_h265_loop(src, os.path.join(tmp, f"r_{tag}_").encode(), n, threads, 1, C.byref(sec))
                return done, sec.value

            ours(8, 1, 0, "warm")
            n1 = 40
            done, sec = ours(n1, 1, 0, "s")
            rec["ms_per_call_1_thread"] = 1000 * sec / n1 if done == n1 else None
            nT = 24 * cores
            done, sec = ours(nT, cores, 0, "t")
            rec["pictures_per_s_threads"] = nT / sec if done == nT else None
            ours(2 * 64 + 8, cores, 64, "warmb")  # the scope's pinned pools and batch encoder are made once and kept
            done, sec = ours(nT, cores, 64, "b")
            rec["pictures_per_s_threads_batch_scope_64"] = nT / sec if done == nT else None
            done, sec = ours(4 * n1, 1, 64, "b1")
            rec["pictures_per_s_1_thread_batch_scope_64"] = 4 * n1 / sec if done == 4 * n1 else None
            same = None
            if ref is not None:
                theirs(4, 1, "warm")
                done, sec = theirs(n1, 1, "s")
                rec["reference_ms_per_call_1_thread"] = 1000 * sec / n1 if done == n1 else None
                done, sec = theirs(nT // 2, cores, "t")
                rec["reference_pictures_per_s_threads"] = (nT // 2) / sec if done == nT // 2 else None
                a, b = os.path.join(tmp, "o_s_0.jpeg"), os.path.join(tmp, "r_s_0.jpeg")
                c = os.path.join(tmp, f"o_b_{nT - 1}.jpeg")
                same = open(a, "rb").read() == open(b, "rb").read() == open(c, "rb").read()
            rec["identical_to_reference_output"] = same
            rec["threads"] = cores
            out["pictures"][name] = rec
    finally:
        import shutil

        shutil.rmtree(tmp, ignore_errors=True)
    return out


def run_ours(a):
    import torch
    import torch.distributed as dist

    import h2j_b200

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the h2j_b200 path has no CPU fallback")
    dev_index, mapping, link_rates = device_plan(torch, local_rank, world)
    torch.cuda.set_device(dev_index)
    dev = torch.device("cuda", dev_index)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cx = Ctx(torch, dist, dev, rank, world)

    w, h = a.width, a.height
    F, SB, NS = a.frames, a.sub_batch or a.frames, a.slots
    assert F % SB == 0 and F % a.e2e_sub_batch == 0
    nsub = F // SB
    lo, hi = h2j_b200.shard_range(world * F, rank, world)  # the job is world*F distinct frames, sharded per image
    assert hi - lo == F
    d_frames, fb, stride = make_frames_torch(F, w, h, dev, seed0=lo)
    torch.cuda.synchronize()
    cores = os.cpu_count() or 1

    enc = h2j_b200.Encoder(max_width=w, max_height=h, max_batch=SB, n_slots=NS, device=dev_index, profile=True,
                           max_jpeg_bytes=a.max_jpeg_bytes)
    streams = [torch.cuda.Stream(device=dev) for _ in range(NS)]
    for s_i, st in enumerate(streams):
        enc.set_stream(s_i, st.cuda_stream)

    # ---- value: device-resident, with a parity sample out of the timed launches ----------------------
    keep = dump_sample(F) if a.dump_outputs and rank == 0 else ()
    dp = device_pass(cx, enc, streams, d_frames, stride, fb, F, SB, NS, w, h, a.steps, a.warmup, a.profile_every, sample=a.parity_frames,
                     keep_frames=keep)
    if keep:
        dump_outputs(a.dump_outputs, dp["last_step"])
    value, dev_ms_max, clocks = dp["value"], dp["dev_ms_max"], dp["clocks"]
    if world > 1:  # every rank's own time and clock, so that a slow GPU (power cap, clocks) shows in the line
        flags = cx.gather(1.0 if clocks.get("reasons") and clocks["reasons"] != ["no samples"] else 0.0)
        clocks["per_rank"] = {"ms_timed_region": [round(x, 3) for x in cx.gather(dp["dev_ms"])], "sm_mhz": cx.gather(clocks.get("sm_mhz") or 0.0),
                              "ranks_with_throttle_reasons": [i for i, x in enumerate(flags) if x > 0]}

    # ---- sustained: the same pass for at least --sustain-seconds ---------------------------------------
    sustained = None
    if a.sustain_seconds > 0:
        sp = device_pass(cx, enc, streams, d_frames, stride, fb, F, SB, NS, w, h, 1, 0, 0, sample=0, min_seconds=a.sustain_seconds)
        sustained = {"value": sp["value"], "unit": UNIT, "seconds": sp["dev_ms_max"] / 1000.0, "steps": sp["steps"], "clocks": sp["clocks"],
                     "note": "same launches as `value`, repeated back to back for the stated time (no per-kernel brackets)"}

    # ---- informational: the same job with two half-batches in flight on two streams ------------------
    # (the HBM-bound K1 and the latency-bound K3 of one half run under the issue-bound kernels of the other; not the
    # headline `value`, whose single stream keeps the per-kernel brackets clean)
    overlap = None
    if not a.no_overlap and NS == 1 and nsub == 1 and F % 2 == 0 and F >= 64:
        try:
            H = F // 2
            enc_o = h2j_b200.Encoder(max_width=w, max_height=h, max_batch=H, n_slots=2, device=dev_index, max_jpeg_bytes=a.max_jpeg_bytes)
            ost = [torch.cuda.Stream(device=dev) for _ in range(2)]
            for s_i, st in enumerate(ost):
                enc_o.set_stream(s_i, st.cuda_stream)
            op = device_pass(cx, enc_o, ost, d_frames, stride, fb, F, H, 2, w, h, a.steps, a.warmup, 0)
            overlap = {"value": op["value"], "unit": UNIT, "slots": 2, "sub_batch": H,
                       "note": "informational: two half-batches in flight on two streams, device-resident, CUDA events"}
            enc_o.close()
        except Exception as ex:
            overlap = {"error": str(ex)}

    # ---- roofline of the dominant kernel ------------------------------------------------------------
    peak, peak_src = hbm_peak()
    dp["avg_image_bytes"] = None
    per_kernel, alg_bytes = kernel_table(dp, w, h, fb, SB, peak)
    dom = max((k for k in per_kernel if k in ("fdct_quant_kernel", "entropy_walk_kernel", "mbvar_kernel", "stuff_kernel", "scan_place_kernel")),
              key=lambda k: per_kernel[k]["avg_ms"])
    traffic, traffic_src = None, None
    try:  # DRAM bytes per frame of the dominant kernel from the committed ncu --set full capture (tools/ncu_traffic.py)
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = tj["kernels"][dom]["dram_bytes_per_frame"] * SB
        traffic_src = f"{tj['source']} ({tj['frames_per_launch']}-frame launch, scaled to {SB})"
    except Exception:
        pass
    step_ms = dev_ms_max / dp["steps"]
    roof = {"bound": "hbm", "kernel": dom, "achieved": per_kernel[dom]["gbs"], "peak": peak, "unit": "GB/s",
            "frac": per_kernel[dom]["gbs"] / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": alg_bytes[dom] * SB, "kernel_share_of_step": per_kernel[dom]["avg_ms"] * nsub / step_ms,
            "note": f"per-kernel CUDA events on the launching stream inside the timed region, on every {max(1, a.profile_every)}-th step "
                    "(one slot: no other stream's kernels inside a bracket)" if NS == 1 else "per-kernel CUDA events on the launching stream; several slots in flight, so a "
                    "bracket can include a neighbour stream's kernels (lower bound on the kernel's own rate)"}
    for k in ("fdct_quant_kernel", "mbvar_kernel", "entropy_walk_kernel"):
        if k in per_kernel and "gbs" in per_kernel[k]:
            roof[k + "_frac"] = per_kernel[k]["gbs"] / peak
    if roof.get("mbvar_kernel_frac", 0) > 1.0:
        roof["mbvar_kernel_note"] = ("read-only kernel: it streams faster than the peak, which was measured with a copy (reads and writes "
                                     "share the bus and pay the read/write turnarounds)")
    # the whole step against the bytes no implementation can avoid: pixels in, JPEG out
    roof["pipeline"] = {"unavoidable_bytes_per_frame": fb + dp["avg_jpeg"], "gbs": (fb + dp["avg_jpeg"]) * value / world / 1e9,
                        "frac": (fb + dp["avg_jpeg"]) * value / world / 1e9 / peak,
                        "note": "frames/s per GPU x (input frame + JPEG) bytes against the HBM peak: every kernel of the step is bound by instruction issue, not by memory"}
    enc.close()

    # ---- e2e: pinned host in, pinned host out ------------------------------------------------------
    e2e = None
    if not a.no_e2e:
        # the job is still world*F frames sharded per image, but a rank's share follows its GPU's host->device rate where the
        # box's links are not equal (a rank behind a slower link would otherwise set the time for everybody)
        e_frames, e_F, shards = d_frames, F, None
        if link_rates and os.environ.get("H2J_BENCH_BALANCE", "1") != "0" and max(link_rates) > 1.05 * min(link_rates):
            shards = h2j_b200.weighted_shards(world * F, link_rates, a.e2e_sub_batch)
            e_lo, e_hi = shards[rank]
            e_F = e_hi - e_lo
            if (e_lo, e_hi) != (lo, hi):
                e_frames, _, _ = make_frames_torch(e_F, w, h, dev, seed0=e_lo)
                torch.cuda.synchronize()
        e2e = e2e_pass(cx, e_frames, stride, fb, e_F, a.e2e_sub_batch, a.e2e_slots, w, h, a.steps, a.warmup, sample=6, job_frames=world * F)
        e2e["rank_to_gpu"] = mapping
        e2e["shards"] = {"frames_per_rank": [hi_ - lo_ for lo_, hi_ in shards], "weights_h2d_gbs": link_rates,
                         "note": "per-image shards in proportion to each GPU's measured host->device rate"} if shards else "equal: F frames per rank"
        if e_frames is not d_frames:
            del e_frames
            torch.cuda.empty_cache()

    # ---- the reference's own call shapes: one picture, and IDecoder::H265ToJpeg (rank 0) -------------
    single, dropin = None, None
    if rank == 0 and not a.no_extras:
        try:
            single = single_frame_record(cx, w, h, d_frames, stride, fb)
        except Exception as ex:
            single = {"error": str(ex)}
        if world == 1:
            try:
                dropin = dropin_record(cores)
            except Exception as ex:
                dropin = {"error": str(ex)}

    # ---- CPU baseline (rank 0, N=1 only) -------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        host8 = d_frames[:8, :fb].cpu().numpy()
        n0 = max(4 * cores, 32)
        dt0, _, _ = cpu_encode_sample(host8, w, h, n0, cores)  # warm + calibrate
        n = a.cpu_frames or max(n0, int(a.cpu_seconds * n0 / dt0))
        dt, kind, _ = cpu_encode_sample(host8, w, h, n, cores)
        cpu = {"value": n / dt, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": f"{n} frames (8 of the bench frames, cycled) on {cores} host threads, {dt:.1f} s of wall time; the reference arm copies each "
                         "frame into a fresh AVFrame and writes its JPEG to a tmpfs file (its stock saveJpegtoFile), which the GPU arm's e2e does not"}

    # ---- BASELINE.json configs[3]: 4K and odd-size frames, outside the headline ----------------------
    others = None
    if not a.no_other_configs:
        del d_frames
        torch.cuda.empty_cache()
        others = []
        for (ow, oh, oF, oESB, ofmt) in ((3840, 2160, 256, 16, 0), (1918, 1078, 512, 64, 0), (1920, 1080, 512, 64, 1), (1920, 1080, 512, 64, 2)):
            try:
                others.append(other_config(cx, ow, oh, oF, oESB, a, chroma_format=ofmt))
            except Exception as ex:
                others.append({"width": ow, "height": oh, "chroma_format": ofmt, "error": str(ex)})

    nv12 = None
    if not a.no_other_configs:
        try:
            nv12 = nv12_record(cx, w, h, 512, a)
        except Exception as ex:
            nv12 = {"error": str(ex)}

    camera = None
    if not a.no_other_configs and world == 1:
        try:
            camera = camera_record(cx, 512, a)
        except Exception as ex:
            camera = {"error": str(ex)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": dp["steps"], "warmup": a.warmup,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/int16", "data": "synthetic",
            "mpixel_per_s": value * w * h / 1e6,
            "config": {"workload": f"{F} distinct synthetic textured {w}x{h} yuv420p frames per GPU per step (configs[2] shape), "
                                   f"sub-batches of {SB} on {NS} streams, bit-exact ffmpeg-mjpeg output; host of this run: {cores} cores "
                                   "(the reference arm and cpu_baseline use all of them; the speed-up against them moves with the core count)",
                       "frames_per_step_per_gpu": F, "sub_batch": SB, "slots": NS,
                       "l2_policy": f"inputs larger than L2: {F * fb / 1e6:.0f} MB of frames per step",
                       "avg_jpeg_bytes": dp["avg_jpeg"], "parity_sampled": dp["parity"], "host_cores": cores, "rank_to_gpu": mapping,
                       "reference_arm_asymmetry": "the reference arm pays a 3.1 MB copy into a fresh AVFrame and a tmpfs file write per frame "
                                                  "(its stock path); the GPU arm's e2e ends in pinned host memory"},
            "clocks": clocks, "e2e": e2e, "sustained": sustained, "two_stream": overlap, "gpu_launches": dp["launches"],
            "wall_ms_per_step": 1000 * dp["wall_s"] / dp["steps"],
            "roofline": roof, "kernels": per_kernel, "cpu_baseline": cpu, "single_frame": single, "dropin": dropin, "other_configs": others, "nv12_device_input": nv12, "camera_content": camera,
        }
        emit_line(line)
    if world > 1:
        dist.barrier()
        if local_rank == 0:  # the device plan of this launch (device_plan) has been read by everybody
            try:
                os.unlink(os.path.join(tempfile.gettempdir(), f"h2j_bench_devices_{os.getppid()}_{os.environ.get('MASTER_PORT', '0')}.json"))
            except OSError:
                pass
        dist.destroy_process_group()


_json_out = None


def emit_line(line):
    print(json.dumps(line), file=_json_out or sys.stdout, flush=True)


def main():
    global _json_out
    a = parse_args()
    # stdout carries exactly ONE line, the JSON: whatever libraries write to file descriptor 1 (NCCL prints its version
    # there) goes to stderr instead
    sys.stdout.flush()
    _json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if a.impl == "reference":
        run_reference_arm(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
