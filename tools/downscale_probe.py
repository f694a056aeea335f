#!/usr/bin/env python
"""Device-resident thumbnails/s of h2j_submit_device_downscaled (DESIGN.md row (f)(7)), 512 x 1080p sources per launch, at
factors 2, 4 and 8, from two source layouts:

  NV12 at a hardware decoder's layout (pitch 2048, pair plane behind 1088 rows)
  I420, tight frames 256-byte aligned (the bench's frames)

alternated with the full-size encode of the same frames (h2j_submit_device_semiplanar read in place, h2j_submit_device).  One
encoder (max 1920x1088, batch 512) serves every variant.  Every variant is warmed up; then rounds of one timed sample per
variant (STEPS submit + collect_device each, CUDA events on the slot's stream) alternate the variants, and the line reports the
median and the spread (min, max).  After every timed sample six frames of its last launch are compared with the oracle's JPEG
of D_k(frame) (tests/support/downscale.py).  The sources (1.7 GB NV12, 1.6 GB I420) are far larger than L2.

A second pass (torch.profiler, CUDA activities) times downscale_list_kernel per factor and layout, and nv12_to_i420_kernel
(a split-first NV12 submit) in the same run, and lists the kernels a uniform downscaled submit ran: the pipeline's batch forms
(LIST = false).  Algorithmic bytes of the downscale: the source's tight frame read + the downscaled tight frame written; of the
split: 2 * fb.  Prints one JSON line (and writes it to --out).  Run on the GPU box: python tools/downscale_probe.py --out FILE"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "h264-h265-to-jpeg_b200")]

import torch  # noqa: E402

import h2j_b200  # noqa: E402
from bench import make_frames_torch  # noqa: E402
from tests.support import oracle as orc  # noqa: E402
from tests.support.downscale import FACTORS, downscale_planar  # noqa: E402

W, H, N = 1920, 1080, 512
ROWS, PITCH = 1088, 2048
PICK = [0, 97, 200, 311, 402, 511]


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def kernel_us(prof, name):
    """mean device time per launch of the kernels whose name contains `name`, in microseconds (None if not captured)"""
    tot, cnt = 0.0, 0
    for ev in prof.key_averages():
        if name in ev.key:
            tot += getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            cnt += ev.count
    return round(tot / cnt, 2) if cnt else None


def tight_bytes(w, h):
    ch, cw = h2j_b200.chroma_shape(w, h, 0)
    return w * h + 2 * cw * ch


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    result = {"what": f"device-resident frames/s, {N} x {W}x{H} sources per launch, {a.steps} launches per sample, {a.rounds} alternated rounds",
              "gpu": gpu_identity(), "variants": {}, "kernels": {}}
    d_i420, fb, stride = make_frames_torch(N, W, H, dev, seed0=9100)
    ch, cw = h2j_b200.chroma_shape(W, H, 0)
    y = d_i420[:, : W * H].view(-1, H, W)
    u = d_i420[:, W * H: W * H + cw * ch].view(-1, ch, cw)
    v = d_i420[:, W * H + cw * ch: fb].view(-1, ch, cw)
    nv12 = torch.full((N, PITCH * ROWS * 3 // 2), 0x5A, dtype=torch.uint8, device=dev)
    nv12[:, : PITCH * H].view(-1, H, PITCH)[:, :, :W] = y
    uv = nv12[:, PITCH * ROWS: PITCH * ROWS + PITCH * ch].view(-1, ch, PITCH)
    uv[:, :, 0:W:2] = u
    uv[:, :, 1:W:2] = v
    nv_stride = nv12.shape[1]
    F = h2j_b200.FrameDesc
    nv_descs = [F(nv12.data_ptr() + i * nv_stride, W, H, PITCH, PITCH, PITCH * ROWS, 0) for i in range(N)]
    i420_descs = [F(d_i420.data_ptr() + i * stride, W, H, W, cw, W * H, W * H + cw * ch) for i in range(N)]
    torch.cuda.synchronize()
    src = {}
    for i in PICK:
        f = d_i420[i, :fb].cpu().numpy()
        src[i] = (f[: W * H].reshape(H, W), f[W * H: W * H + cw * ch].reshape(ch, cw), f[W * H + cw * ch:].reshape(ch, cw))
    want = {k: {i: orc.oracle_encode(*(downscale_planar(*src[i], k) if k > 1 else src[i]))[0] for i in PICK} for k in (1,) + FACTORS}

    enc = h2j_b200.Encoder(max_width=W, max_height=ROWS, max_batch=N, n_slots=1, max_jpeg_bytes=4 * 1024 * 1024)
    st = torch.cuda.Stream(device=dev)
    enc.set_stream(0, st.cuda_stream)
    variants = {  # name -> (submit, factor of the oracle's picture)
        "nv12_full_in_place": (lambda: enc.submit_device_semiplanar(0, nv12.data_ptr(), nv_stride, PITCH, PITCH * ROWS, N, W, H), 1),
        "i420_full": (lambda: enc.submit_device(0, d_i420.data_ptr(), stride, N, W, H), 1),
    }
    for k in FACTORS:
        variants[f"nv12_k{k}"] = ((lambda k=k: enc.submit_device_downscaled(0, h2j_b200.LAYOUT_SEMIPLANAR, nv_descs, k)), k)
        variants[f"i420_k{k}"] = ((lambda k=k: enc.submit_device_downscaled(0, h2j_b200.LAYOUT_PLANAR, i420_descs, k)), k)
    samples = {k: [] for k in variants}
    parity = {k: [] for k in variants}
    launches = {}
    for name, (go, _) in variants.items():  # warm-up, and the launches one batch takes
        before = enc.kernel_launches
        go()
        enc.collect_device(0)
        launches[name] = enc.kernel_launches - before
        go()
        enc.collect_device(0)
    for _ in range(a.rounds):
        for name, (go, k) in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(a.steps):
                go()
                d_out, cap, sizes, status = enc.collect_device(0)
            e1.record(st)
            e1.synchronize()
            samples[name].append(N * a.steps / (e0.elapsed_time(e1) / 1000.0))
            bad = [i for i in PICK if int(status[i]) != 0 or enc.read_device(d_out + i * cap, int(sizes[i])) != want[k][i]]
            parity[name].append(not bad)
    for name in variants:
        s = samples[name]
        result["variants"][name] = {"frames_per_s_median": round(statistics.median(s)), "min": round(min(s)), "max": round(max(s)),
                                    "kernel_launches_per_batch": launches[name], "parity_6_frames_every_round": all(parity[name])}
    vv = result["variants"]
    result["thumbnail_over_full"] = {f"{lay}_k{k}": round(vv[f"{lay}_k{k}"]["frames_per_s_median"] / vv[full]["frames_per_s_median"], 3)
                                     for lay, full in (("nv12", "nv12_full_in_place"), ("i420", "i420_full")) for k in FACTORS}

    # kernel times and names, in a run of their own
    from torch.profiler import ProfilerActivity, profile

    def profiled(go):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                go()
                enc.collect_device(0)
            torch.cuda.synchronize()
        return prof

    for lay in ("nv12", "i420"):
        for k in FACTORS:
            prof = profiled(variants[f"{lay}_k{k}"][0])
            us = kernel_us(prof, "downscale_list_kernel")
            dw, dh = h2j_b200.downscaled_size(W, H, k)
            moved = (fb + tight_bytes(dw, dh)) * N
            entry = {"us_per_launch_of_512": us, "bytes_per_launch": moved, "algorithmic_GB_per_s": round(moved / us / 1e3, 1) if us else None}
            if k == 4:
                entry["kernels_ran"] = sorted({ev.key.split("(")[0] for ev in prof.key_averages() if "h2j::" in ev.key})
            result["kernels"][f"downscale_{lay}_k{k}"] = entry

    def split_first():
        enc.set_knob("semiplanar_prepass", 1)
        enc.submit_device_semiplanar(0, nv12.data_ptr(), nv_stride, PITCH, PITCH * ROWS, N, W, H)
        enc.set_knob("semiplanar_prepass", 0)

    prof = profiled(split_first)
    us = kernel_us(prof, "nv12_to_i420_kernel")
    result["kernels"]["nv12_to_i420_kernel"] = {"us_per_launch_of_512": us, "bytes_per_launch": 2 * fb * N,
                                                "algorithmic_GB_per_s": round(2 * fb * N / us / 1e3, 1) if us else None}
    split = result["kernels"]["nv12_to_i420_kernel"]["algorithmic_GB_per_s"]
    result["downscale_k2_rate_over_split"] = {lay: round(result["kernels"][f"downscale_{lay}_k2"]["algorithmic_GB_per_s"] / split, 3)
                                              for lay in ("nv12", "i420")}
    enc.close()
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not all(x["parity_6_frames_every_round"] for x in vv.values()):
        sys.exit(1)


if __name__ == "__main__":
    main()
