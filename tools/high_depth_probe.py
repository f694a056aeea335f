#!/usr/bin/env python
"""Device-resident throughput of high-bit-depth input (DESIGN.md row (f)(5)) against the 8-bit layouts, 512 x 1080p per launch:

  4:2:0  P010 (h2j_submit_device_semiplanar16, bit_depth 16), NV12 read in place, I420 (h2j_submit_device)
  4:2:2  P216 (semiplanar16), NV16 read in place
  4:4:4  16-bit planar at a decoder's surface layout (h2j_submit_device_pitched16, bit_depth 16), 8-bit at the same layout

Decoder layouts: pitch rounded up to 256 bytes, planes behind 1088 rows.  The 16-bit words are the 8-bit frame's samples in the
high byte and random bits in the low byte, so every variant of a format encodes the same pictures.  Every variant is warmed up;
then rounds of one timed sample per variant (STEPS submit + collect_device each, CUDA events on the slot's stream) alternate the
variants, and the line reports the median and the spread (min, max) of frames/s.  After every timed sample six frames of its
last launch are compared with the oracle's JPEG of the 8-bit planar frame.  The input (3 GB and more per 16-bit variant) is
far larger than L2.

A second pass (torch.profiler, CUDA activities) times depth_to_8_kernel and, from a split-first NV12 submit,
nv12_to_i420_kernel.  Algorithmic rate: the conversion reads 2 * fb and writes fb bytes per frame, the split reads and writes
fb (fb: the tight 8-bit frame).  Last, the single-picture call time of h2j_encode_frame16 against h2j_encode_frame at 1080p
(pageable planes, alternated).  Prints one JSON line (and writes it to --out).  Run on the GPU box:
python tools/high_depth_probe.py --out FILE"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "h264-h265-to-jpeg_b200")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import h2j_b200  # noqa: E402
from bench import make_frames_torch  # noqa: E402
from tests.support import oracle as orc  # noqa: E402

W, H, N = 1920, 1080, 512
ROWS = 1088
PICK = [0, 97, 200, 311, 402, 511]


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def planes_of(d, fmt):
    """(n, fb) planar frames -> [y, u, v] views (n, rows, cols)"""
    ch, cw = h2j_b200.chroma_shape(W, H, fmt)
    return [d[:, : W * H].view(-1, H, W), d[:, W * H: W * H + cw * ch].view(-1, ch, cw), d[:, W * H + cw * ch: W * H + 2 * cw * ch].view(-1, ch, cw)]


def widen(p, g):
    """8-bit samples in the high byte, random low byte (as int16: the same 16 bits)"""
    x = p.to(torch.int32) << 8 | torch.randint(0, 256, p.shape, device=p.device, generator=g, dtype=torch.int32)
    return (x - ((x >> 15) << 16)).to(torch.int16)


def semiplanar(d, fmt, bps, g):
    """-> (frames, frame stride, pitch, uv_offset), bytes; bps = bytes per sample"""
    y, u, v = planes_of(d, fmt)
    ch, cw = u.shape[1:]
    pitch = (bps * max(W, 2 * cw) + 255) // 256 * 256
    stride = pitch * ROWS + pitch * ch
    out = torch.full((d.shape[0], stride // bps), 0x5A5A if bps == 2 else 0x5A, dtype=torch.int16 if bps == 2 else torch.uint8, device=d.device)
    cvt = (lambda p: widen(p, g)) if bps == 2 else (lambda p: p)
    pp = pitch // bps
    out[:, : pp * H].view(-1, H, pp)[:, :, :W] = cvt(y)
    uv = out[:, pp * ROWS: pp * ROWS + pp * ch].view(-1, ch, pp)
    uv[:, :, 0: 2 * cw: 2] = cvt(u)
    uv[:, :, 1: 2 * cw: 2] = cvt(v)
    return out, stride, pitch, pitch * ROWS


def surface(d, fmt, bps, g):
    """planar frames at a decoder's surface layout -> (frames, stride, pitch): planes at multiples of pitch * 1088"""
    planes = planes_of(d, fmt)
    pitch = (bps * W + 255) // 256 * 256
    stride = 3 * pitch * ROWS
    out = torch.zeros((d.shape[0], stride // bps), dtype=torch.int16 if bps == 2 else torch.uint8, device=d.device)
    pp = pitch // bps
    for k, p in enumerate(planes):
        out[:, k * pp * ROWS: k * pp * ROWS + pp * p.shape[1]].view(-1, p.shape[1], pp)[:, :, : p.shape[2]] = widen(p, g) if bps == 2 else p
    return out, stride, pitch


def kernel_us(prof, name):
    """mean device time per launch of the kernels whose name contains `name`, in microseconds (None if not captured)"""
    tot, cnt = 0.0, 0
    for ev in prof.key_averages():
        if name in ev.key:
            tot += getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            cnt += ev.count
    return round(tot / cnt, 2) if cnt else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--single-calls", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    result = {"what": f"device-resident frames/s, {N} x {W}x{H} per launch, {a.steps} launches per sample, {a.rounds} alternated rounds",
              "gpu": gpu_identity(), "variants": {}, "kernels": {}}
    for fmt, tag in ((0, "420"), (1, "422"), (2, "444")):
        d_planar, fb, pstride = make_frames_torch(N, W, H, dev, seed0=7000 + fmt, chroma_format=fmt)
        ch, cw = h2j_b200.chroma_shape(W, H, fmt)
        want = {}
        for i in PICK:
            f = d_planar[i, :fb].cpu().numpy()
            want[i] = orc.oracle_encode(f[: W * H].reshape(H, W), f[W * H: W * H + cw * ch].reshape(ch, cw),
                                        f[W * H + cw * ch: fb].reshape(ch, cw), chroma_format=fmt)[0]
        enc = h2j_b200.Encoder(max_width=W, max_height=H, max_batch=N, n_slots=1, chroma_format=fmt, max_jpeg_bytes=4 * 1024 * 1024)
        st = torch.cuda.Stream(device=dev)
        enc.set_stream(0, st.cuda_stream)
        keep = []
        if fmt in (0, 1):
            s16, st16, p16, uv16 = semiplanar(d_planar, fmt, 2, g)
            s8, st8, p8, uv8 = semiplanar(d_planar, fmt, 1, g)
            keep += [s16, s8]
            n16, n8 = ("p010", "nv12") if fmt == 0 else ("p216", "nv16")

            def sp8(prepass):
                def go():
                    enc.set_knob("semiplanar_prepass", prepass)
                    enc.submit_device_semiplanar(0, s8.data_ptr(), st8, p8, uv8, N, W, H)
                return go

            variants = {f"{n16}_semiplanar16": lambda: enc.submit_device_semiplanar16(0, s16.data_ptr(), st16, p16, uv16, 16, N, W, H),
                        f"{n8}_in_place": sp8(0)}
            if fmt == 0:
                variants["i420_planar"] = lambda: enc.submit_device(0, d_planar.data_ptr(), pstride, N, W, H)
            profiled = {f"{n16}_semiplanar16": variants[f"{n16}_semiplanar16"], f"{n8}_split_first": sp8(1)}
        else:
            s16, st16, p16 = surface(d_planar, fmt, 2, g)
            s8, st8, p8 = surface(d_planar, fmt, 1, g)
            keep += [s16, s8]
            variants = {"444_pitched16_decoder_layout": lambda: enc.submit_device_pitched16(0, s16.data_ptr(), st16, p16, p16, p16 * ROWS,
                                                                                             2 * p16 * ROWS, 16, N, W, H),
                        "444_pitched8_decoder_layout": lambda: enc.submit_device_pitched(0, s8.data_ptr(), st8, p8, p8, p8 * ROWS,
                                                                                          2 * p8 * ROWS, N, W, H)}
            profiled = {"444_pitched16_decoder_layout": variants["444_pitched16_decoder_layout"]}
        torch.cuda.synchronize()
        samples = {k: [] for k in variants}
        parity = {k: [] for k in variants}
        launches = {}
        for k, go in variants.items():  # warm-up, and the launches one batch takes
            before = enc.kernel_launches
            go()
            enc.collect_device(0)
            launches[k] = enc.kernel_launches - before
            go()
            enc.collect_device(0)
        for _ in range(a.rounds):
            for k, go in variants.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                for _ in range(a.steps):
                    go()
                    d_out, cap, sizes, status = enc.collect_device(0)
                e1.record(st)
                e1.synchronize()
                samples[k].append(N * a.steps / (e0.elapsed_time(e1) / 1000.0))
                bad = [i for i in PICK if int(status[i]) != 0 or enc.read_device(d_out + i * cap, int(sizes[i])) != want[i]]
                parity[k].append(not bad)
        for k in variants:
            s = samples[k]
            result["variants"][k] = {"frames_per_s_median": round(statistics.median(s)), "min": round(min(s)), "max": round(max(s)),
                                     "kernel_launches_per_batch": launches[k], "parity_6_frames_every_round": all(parity[k])}
        # kernel times, in a run of their own
        from torch.profiler import ProfilerActivity, profile

        for k, go in profiled.items():
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    go()
                    enc.collect_device(0)
                torch.cuda.synchronize()
            kname = "nv12_to_i420_kernel" if k.endswith("split_first") else "depth_to_8_kernel"
            us = kernel_us(prof, kname)
            moved = (2 if kname == "nv12_to_i420_kernel" else 3) * fb * N
            result["kernels"][f"{tag}_{kname}"] = {"variant": k, "us_per_launch_of_512": us, "bytes_per_launch": moved,
                                                     "algorithmic_GB_per_s": round(moved / us / 1e3, 1) if us else None}
        enc.close()
        del keep, s16, s8, d_planar
        torch.cuda.empty_cache()

    # single-picture call time at 1080p, 4:2:0, pageable planes
    y, u, v = orc.synth_planes(W, H, "textured", seed=5, amp=30)
    rng = np.random.default_rng(5)
    y16, u16, v16 = [(x.astype(np.uint16) << 8) | rng.integers(0, 256, x.shape, dtype=np.uint16) for x in (y, u, v)]
    want = orc.oracle_encode(y, u, v)[0]
    with h2j_b200.Encoder(max_width=W, max_height=H, max_batch=1, n_slots=1) as e:
        out = np.empty(e.out_capacity, np.uint8)
        n = C.c_size_t(0)

        def args(ps):
            return (C.c_void_p * 3)(*(p.ctypes.data for p in ps)), (C.c_int * 3)(*(p.strides[0] for p in ps))

        a8, a16 = args((y, u, v)), args((y16, u16, v16))
        calls = {"h2j_encode_frame": lambda: e._lib.h2j_encode_frame(e._h, a8[0], a8[1], W, H, out.ctypes.data, out.size, C.byref(n)),
                 "h2j_encode_frame16": lambda: e._lib.h2j_encode_frame16(e._h, a16[0], a16[1], 16, W, H, out.ctypes.data, out.size, C.byref(n))}
        times = {k: [] for k in calls}
        for k, c in calls.items():
            for _ in range(5):
                assert c() == 0
            assert out[: n.value].tobytes() == want, k
        for _ in range(a.single_calls):
            for k, c in calls.items():
                t0 = time.perf_counter()
                rc = c()
                times[k].append((time.perf_counter() - t0) * 1e3)
                assert rc == 0
        result["single_picture_ms_median"] = {k: round(statistics.median(t), 3) for k, t in times.items()}
        result["single_picture_parity"] = out[: n.value].tobytes() == want
    v = result["variants"]
    result["high_depth_over_8bit"] = {"p010_over_nv12_in_place": round(v["p010_semiplanar16"]["frames_per_s_median"] / v["nv12_in_place"]["frames_per_s_median"], 3),
                                      "p010_over_i420": round(v["p010_semiplanar16"]["frames_per_s_median"] / v["i420_planar"]["frames_per_s_median"], 3),
                                      "p216_over_nv16_in_place": round(v["p216_semiplanar16"]["frames_per_s_median"] / v["nv16_in_place"]["frames_per_s_median"], 3),
                                      "444_16_over_8": round(v["444_pitched16_decoder_layout"]["frames_per_s_median"] / v["444_pitched8_decoder_layout"]["frames_per_s_median"], 3)}
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not all(x["parity_6_frames_every_round"] for x in v.values()) or not result["single_picture_parity"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
