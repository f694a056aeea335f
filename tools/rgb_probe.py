#!/usr/bin/env python
"""Device-resident frames/s of h2j_submit_device_rgb (DESIGN.md row (f)(8)), 512 x 1080p frames per launch, from

  RGB24, tight rows (5760 bytes)               at 4:2:0 and at 4:4:4
  BGRX at a pitch of 7680 bytes (RGBA8 surface) at 4:2:0
  planar CHW (torch (3, H, W))                 at 4:2:0

alternated with h2j_submit_device of the converted planar frames C(frame) (the I420 / 4:4:4 frames a caller would have to
make first).  One encoder per chroma format (max 1920x1088, batch 512) serves its variants.  Every variant is warmed up;
then rounds of one timed sample per variant (STEPS submit + collect_device each, CUDA events on the slot's stream) alternate
the variants, and the line reports the median and the spread (min, max).  After every timed sample six frames of its last
launch are compared with the oracle's JPEG of C(frame) (tests/support/rgb.py).  Every source set is larger than L2.

A second pass (torch.profiler, CUDA activities) times rgb_to_planar_kernel per variant, with nv12_to_i420_kernel (a
split-first NV12 submit of the same frames) in the same run as the yardstick.  Algorithmic bytes of the conversion: the
source's pixels read + the tight planar frame written; of the split: 2 * fb.  A third pass times h2j_encode_frame_rgb of a
1080p RGB24 picture in pageable memory against h2j_encode_frame of its I420 frame, alternated.  Prints one JSON line (and
writes it to --out).  Run on the GPU box: python tools/rgb_probe.py --out FILE"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "h264-h265-to-jpeg_b200")]

import torch  # noqa: E402

import h2j_b200  # noqa: E402
from bench import make_frames_torch  # noqa: E402
from tests.support import oracle as orc  # noqa: E402
from tests.support import rgb as R  # noqa: E402

W, H, N = 1920, 1080, 512
BGRX_PITCH = 7680
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


def converted(rgb, cf, chunk=32):
    """C(frame) of an (n, H, W, 3) uint8 CUDA tensor as tight planar frames (n, fb) on the device (H and W even: full boxes)"""
    out = []
    for c in rgb.split(chunk):
        r, g, b = (c[..., k].to(torch.int32) for k in range(3))
        y = (R.Y_R * r + R.Y_G * g + R.Y_B * b + 32768) >> 16
        cb = (-R.CB_R * r - R.CB_G * g + R.HALF * b + (128 << 16) + 32767) >> 16
        cr = (R.HALF * r - R.CR_G * g - R.CR_B * b + (128 << 16) + 32767) >> 16
        if cf == 0:
            n = c.shape[0]
            cb = (cb.view(n, H // 2, 2, W // 2, 2).sum((2, 4)) + 2) >> 2
            cr = (cr.view(n, H // 2, 2, W // 2, 2).sum((2, 4)) + 2) >> 2
        out.append(torch.cat([p.reshape(c.shape[0], -1) for p in (y, cb, cr)], 1).to(torch.uint8))
    return torch.cat(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--host-calls", type=int, default=40)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    result = {"what": f"device-resident frames/s, {N} x {W}x{H} frames per launch, {a.steps} launches per sample, {a.rounds} alternated rounds",
              "gpu": gpu_identity(), "variants": {}, "kernels": {}}
    # R, G and B: the luma planes of three textured frame sets
    planes = [make_frames_torch(N, W, H, dev, seed0=9300 + 1000 * k)[0][:, : W * H].view(N, H, W) for k in range(3)]
    rgb = torch.stack(planes, -1).contiguous()  # (N, H, W, 3): RGB24, tight
    del planes
    bgrx = torch.randint(0, 256, (N, H, BGRX_PITCH), dtype=torch.uint8, device=dev)  # the X bytes and the pitch's tail: noise
    bgrx.view(N, H, BGRX_PITCH // 4, 4)[:, :, :W, :3] = rgb.flip(-1)
    chw = rgb.permute(0, 3, 1, 2).contiguous()
    F = h2j_b200.FrameDesc
    src = {
        "rgb24": (h2j_b200.RGB_RGB24, [F(rgb.data_ptr() + i * 3 * W * H, W, H, 3 * W, 0, 0, 0) for i in range(N)], 3 * W * H),
        "bgrx_pitch7680": (h2j_b200.RGB_BGRX, [F(bgrx.data_ptr() + i * BGRX_PITCH * H, W, H, BGRX_PITCH, 0, 0, 0) for i in range(N)], 4 * W * H),
        "planar_chw": (h2j_b200.RGB_PLANAR, [F(chw.data_ptr() + i * 3 * W * H, W, H, W, 0, W * H, 2 * W * H) for i in range(N)], 3 * W * H),
    }
    host_rgb = {i: rgb[i].cpu().numpy() for i in PICK}
    want = {cf: {i: orc.oracle_encode(*R.to_planar(host_rgb[i], R.RGB24, cf), chroma_format=cf)[0] for i in PICK} for cf in (0, 2)}
    yuv = {cf: converted(rgb, cf) for cf in (0, 2)}
    torch.cuda.synchronize()

    encs, variants = {}, {}  # name -> (encoder, submit, chroma format)
    for cf in (0, 2):
        e = h2j_b200.Encoder(max_width=W, max_height=1088, max_batch=N, n_slots=1, max_jpeg_bytes=4 * 1024 * 1024, chroma_format=cf)
        st = torch.cuda.Stream(device=dev)
        e.set_stream(0, st.cuda_stream)
        encs[cf] = (e, st)
        tag = "420" if cf == 0 else "444"
        fb = yuv[cf].shape[1]
        variants[f"planar_{tag}_submit_device"] = (cf, lambda e=e, cf=cf, fb=fb: e.submit_device(0, yuv[cf].data_ptr(), fb, N, W, H))
        for name, (fmt, descs, _) in src.items():
            if cf == 0 or name == "rgb24":
                variants[f"{name}_{tag}"] = (cf, lambda e=e, fmt=fmt, descs=descs: e.submit_device_rgb(0, fmt, descs))
    samples = {k: [] for k in variants}
    parity = {k: [] for k in variants}
    launches = {}
    for name, (cf, go) in variants.items():  # warm-up, and the launches one batch takes
        e = encs[cf][0]
        before = e.kernel_launches
        go()
        e.collect_device(0)
        launches[name] = e.kernel_launches - before
        go()
        e.collect_device(0)
    for _ in range(a.rounds):
        for name, (cf, go) in variants.items():
            e, st = encs[cf]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(a.steps):
                go()
                d_out, cap, sizes, status = e.collect_device(0)
            e1.record(st)
            e1.synchronize()
            samples[name].append(N * a.steps / (e0.elapsed_time(e1) / 1000.0))
            bad = [i for i in PICK if int(status[i]) != 0 or e.read_device(d_out + i * cap, int(sizes[i])) != want[cf][i]]
            parity[name].append(not bad)
    for name in variants:
        s = samples[name]
        result["variants"][name] = {"frames_per_s_median": round(statistics.median(s)), "min": round(min(s)), "max": round(max(s)),
                                    "kernel_launches_per_batch": launches[name], "parity_6_frames_every_round": all(parity[name])}
    vv = result["variants"]
    result["rgb_over_planar_submit"] = {name: round(vv[name]["frames_per_s_median"] / vv[f"planar_{name[-3:]}_submit_device"]["frames_per_s_median"], 3)
                                        for name in vv if not name.startswith("planar_") or name == "planar_chw_420"}

    # kernel times, in a run of their own
    from torch.profiler import ProfilerActivity, profile

    def profiled(e, go):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                go()
                e.collect_device(0)
            torch.cuda.synchronize()
        return prof

    for name, (cf, go) in variants.items():
        if name.startswith("planar_") and name != "planar_chw_420":
            continue
        prof = profiled(encs[cf][0], go)
        us = kernel_us(prof, "rgb_to_planar_kernel")
        moved = (src[name.rsplit("_", 1)[0]][2] + yuv[cf].shape[1]) * N
        result["kernels"][f"rgb_to_planar_{name}"] = {"us_per_launch_of_512": us, "bytes_per_launch": moved,
                                                      "algorithmic_GB_per_s": round(moved / us / 1e3, 1) if us else None}
    # the yardstick: the NV12 split of the same I420 frames
    e = encs[0][0]
    fb0 = yuv[0].shape[1]
    ch, cw = H // 2, W // 2
    nv12 = torch.empty((N, W * H * 3 // 2), dtype=torch.uint8, device=dev)
    nv12[:, : W * H] = yuv[0][:, : W * H]
    uv = nv12[:, W * H:].view(N, ch, W)
    uv[:, :, 0::2] = yuv[0][:, W * H: W * H + cw * ch].view(N, ch, cw)
    uv[:, :, 1::2] = yuv[0][:, W * H + cw * ch:].view(N, ch, cw)
    torch.cuda.synchronize()

    def split_first():
        e.set_knob("semiplanar_prepass", 1)
        e.submit_device_semiplanar(0, nv12.data_ptr(), nv12.shape[1], W, W * H, N, W, H)
        e.set_knob("semiplanar_prepass", 0)

    prof = profiled(e, split_first)
    us = kernel_us(prof, "nv12_to_i420_kernel")
    result["kernels"]["nv12_to_i420_kernel"] = {"us_per_launch_of_512": us, "bytes_per_launch": 2 * fb0 * N,
                                                "algorithmic_GB_per_s": round(2 * fb0 * N / us / 1e3, 1) if us else None}
    split = result["kernels"]["nv12_to_i420_kernel"]["algorithmic_GB_per_s"]
    result["rgb_rate_over_split"] = {k: round(v["algorithmic_GB_per_s"] / split, 3) for k, v in result["kernels"].items() if k.startswith("rgb_")}

    # one picture from pageable host memory: h2j_encode_frame_rgb against h2j_encode_frame, alternated
    i0 = PICK[1]
    pic = host_rgb[i0].copy()
    f = yuv[0][i0].cpu().numpy()
    y, u, v = f[: W * H].reshape(H, W), f[W * H: W * H + cw * ch].reshape(ch, cw), f[W * H + cw * ch:].reshape(ch, cw)
    assert e.rgb2jpeg(pic, h2j_b200.RGB_RGB24) == want[0][i0] and e.yuv2jpeg(y, u, v) == want[0][i0]
    host = {"encode_frame_rgb_rgb24": lambda: e.rgb2jpeg(pic, h2j_b200.RGB_RGB24), "encode_frame_i420": lambda: e.yuv2jpeg(y, u, v)}
    ms = {k: [] for k in host}
    for _ in range(a.rounds):
        for k, go in host.items():
            t0 = time.perf_counter()
            for _ in range(a.host_calls):
                go()
            ms[k].append((time.perf_counter() - t0) * 1000.0 / a.host_calls)
    result["host_1080p_pageable_ms_per_call"] = {k: {"median": round(statistics.median(s), 3), "min": round(min(s), 3), "max": round(max(s), 3)}
                                                 for k, s in ms.items()}
    for e, _ in encs.values():
        e.close()
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fo:
            fo.write(line + "\n")
    if not all(x["parity_6_frames_every_round"] for x in vv.values()):
        sys.exit(1)


if __name__ == "__main__":
    main()
