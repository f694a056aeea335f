#!/usr/bin/env python
"""Device-resident frames/s of h2j_submit_device_resized (DESIGN.md row (f)(9)), 512 x 1080p sources per launch, from two
source layouts:

  NV12 at a hardware decoder's layout (pitch 2048, pair plane behind 1088 rows)
  I420, tight frames 256-byte aligned (the bench's frames)

Variants: BOX, BILINEAR and BICUBIC at 960x540, 1280x720, 640x360, 224x224 and 320x180; an upscale of 960x540 sources to
1920x1080 (BILINEAR); and h2j_submit_device_downscaled at factors 2 and 8 (960x540, 240x135), the box filter at equal output
sizes.  One encoder (max 1920x1088, batch 512) serves every variant.  Every variant is warmed up; then rounds of one timed
sample per variant (STEPS submit + collect_device each, CUDA events on the slot's stream) alternate the variants, and the line
reports the median and the spread (min, max).  After the last round three frames of each variant's last launch are compared
with the oracle's JPEG of the model's planes (tests/support/resize.py).  The sources (1.7 GB NV12, 1.6 GB I420) are far
larger than L2.

A second pass (torch.profiler, CUDA activities) times resize_list_kernel per variant, downscale_list_kernel at factor 2 and
nv12_to_i420_kernel (a split-first NV12 submit).  Algorithmic bytes of a resize or downscale: the source's tight frame read
+ the output's tight frame written; of the split: 2 * fb.  Prints one JSON line (and writes it to --out).  Run on the GPU box:
python tools/resize_probe.py --out FILE"""
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
from tests.support.downscale import downscale_planar  # noqa: E402
from tests.support.resize import resize_planar  # noqa: E402

W, H, N = 1920, 1080, 512
ROWS, PITCH = 1088, 2048
PICK = [0, 257, 511]
SIZES = [(960, 540), (1280, 720), (640, 360), (224, 224), (320, 180)]
FILTERS = {"box": h2j_b200.FILTER_BOX, "bilinear": h2j_b200.FILTER_BILINEAR, "bicubic": h2j_b200.FILTER_BICUBIC}


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
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    result = {"what": f"device-resident frames/s, {N} x {W}x{H} sources per launch, {a.steps} launches per sample, {a.rounds} alternated rounds",
              "gpu": gpu_identity(), "variants": {}, "kernels": {}}
    d_i420, fb, stride = make_frames_torch(N, W, H, dev, seed0=9300)
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
    # 960x540 I420 sources for the upscale: the first 960x540 of every frame's planes, at the frames' pitches
    half = [F(d_i420.data_ptr() + i * stride, 960, 540, W, cw, W * H, W * H + cw * ch) for i in range(N)]
    torch.cuda.synchronize()
    src = {}
    for i in PICK:
        f = d_i420[i, :fb].cpu().numpy()
        src[i] = (f[: W * H].reshape(H, W), f[W * H: W * H + cw * ch].reshape(ch, cw), f[W * H + cw * ch:].reshape(ch, cw))

    enc = h2j_b200.Encoder(max_width=W, max_height=ROWS, max_batch=N, n_slots=1, max_jpeg_bytes=4 * 1024 * 1024)
    st = torch.cuda.Stream(device=dev)
    enc.set_stream(0, st.cuda_stream)
    R, P = h2j_b200.LAYOUT_SEMIPLANAR, h2j_b200.LAYOUT_PLANAR
    variants = {}  # name -> (submit, the model of frame i's planes)
    for lay, descs, layout in (("nv12", nv_descs, R), ("i420", i420_descs, P)):
        for fname, flt in FILTERS.items():
            for ow, oh in SIZES:
                variants[f"{lay}_{fname}_{ow}x{oh}"] = (
                    (lambda d=descs, lo=layout, s=(ow, oh), f=flt: enc.submit_device_resized(0, lo, d, [s] * N, f)),
                    (lambda i, s=(ow, oh), f=flt: resize_planar(*src[i], *s, 0, f)))
        for k in (2, 8):
            variants[f"{lay}_downscaled_k{k}"] = ((lambda d=descs, lo=layout, k=k: enc.submit_device_downscaled(0, lo, d, k)),
                                                  (lambda i, k=k: downscale_planar(*src[i], k)))
    variants["i420_bilinear_960x540_to_1920x1080"] = (
        (lambda: enc.submit_device_resized(0, P, half, [(W, H)] * N, h2j_b200.FILTER_BILINEAR)),
        (lambda i: resize_planar(src[i][0][:540, :960], src[i][1][:270, :480], src[i][2][:270, :480], W, H, 0, 1)))
    samples = {k: [] for k in variants}
    launches = {}
    for name, (go, _) in variants.items():  # warm-up, and the launches one batch takes
        before = enc.kernel_launches
        go()
        enc.collect_device(0)
        launches[name] = enc.kernel_launches - before
    for r in range(a.rounds):
        for name, (go, model) in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(a.steps):
                go()
                d_out, cap, sizes, status = enc.collect_device(0)
            e1.record(st)
            e1.synchronize()
            samples[name].append(N * a.steps / (e0.elapsed_time(e1) / 1000.0))
            if r == a.rounds - 1:
                bad = [i for i in PICK if int(status[i]) != 0 or enc.read_device(d_out + i * cap, int(sizes[i])) != orc.oracle_encode(*model(i))[0]]
                result["variants"][name] = {"parity_3_frames_last_round": not bad}
    for name in variants:
        s = samples[name]
        result["variants"][name].update({"frames_per_s_median": round(statistics.median(s)), "min": round(min(s)), "max": round(max(s)),
                                         "kernel_launches_per_batch": launches[name]})

    from torch.profiler import ProfilerActivity, profile

    def profiled(go):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                go()
                enc.collect_device(0)
            torch.cuda.synchronize()
        return prof

    for name, (go, _) in variants.items():
        kern = "downscale_list_kernel" if "downscaled" in name else "resize_list_kernel"
        prof = profiled(go)
        us = kernel_us(prof, kern)
        if "downscaled" in name:
            out = h2j_b200.downscaled_size(W, H, int(name[-1]))
        else:
            out = tuple(int(x) for x in name.split("_")[-1].split("x"))
        src_bytes = tight_bytes(960, 540) if "to_1920" in name else fb
        moved = (src_bytes + tight_bytes(*out)) * N
        result["kernels"][name] = {"kernel": kern, "us_per_launch_of_512": us, "bytes_per_launch": moved,
                                   "algorithmic_GB_per_s": round(moved / us / 1e3, 1) if us else None}

    def split_first():
        enc.set_knob("semiplanar_prepass", 1)
        enc.submit_device_semiplanar(0, nv12.data_ptr(), nv_stride, PITCH, PITCH * ROWS, N, W, H)
        enc.set_knob("semiplanar_prepass", 0)

    prof = profiled(split_first)
    us = kernel_us(prof, "nv12_to_i420_kernel")
    result["kernels"]["nv12_to_i420_kernel"] = {"us_per_launch_of_512": us, "bytes_per_launch": 2 * fb * N,
                                                "algorithmic_GB_per_s": round(2 * fb * N / us / 1e3, 1) if us else None}
    enc.close()
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not all(x["parity_3_frames_last_round"] for x in result["variants"].values()):
        sys.exit(1)


if __name__ == "__main__":
    main()
