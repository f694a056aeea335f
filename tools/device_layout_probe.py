#!/usr/bin/env python
"""Device-resident throughput of the 4:2:2 / 4:4:4 input layouts (DESIGN.md row (f)(4)), 512 x 1080p frames per launch:

  4:2:2  planar (h2j_submit_device), NV16 read in place, NV16 split first (the prepass)
  4:4:4  planar, NV24 read in place, NV24 split first, planar at a hardware decoder's surface layout (h2j_submit_device_pitched)

Semi-planar frames sit at a decoder's layout: pitch 2048 (NV16) / 4096 (NV24: 3840 bytes of pairs a row), pair plane behind
1088 luma rows.  The pitched frames have one pitch of 2048 and the chroma planes at 2048 * 1088 and 2 * 2048 * 1088.
Every variant is warmed up; then rounds of one timed sample
per variant (STEPS submit + collect_device each, CUDA events on the slot's stream) alternate the variants, and the line reports
the median and the spread (min, max) of frames/s over the rounds.  After every timed sample six frames of its last launch are
compared with the oracle's JPEG of the planar frame.  The working set (2 GB and more per variant) is far larger than L2.
Prints one JSON line (and writes it to --out).  Run on the GPU box: python tools/device_layout_probe.py --out FILE"""
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

W, H, N = 1920, 1080, 512
PITCH, ROWS = 2048, 1088  # a decoder surface: 256-byte aligned pitch, 16-row aligned height


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def semiplanar(d, fmt):
    """-> (frames, frame stride, pitch): the pitch holds a row of pairs (NV24: 2 * 1920 bytes -> 4096)"""
    ch, cw = h2j_b200.chroma_shape(W, H, fmt)
    pitch = (max(W, 2 * cw) + 255) // 256 * 256
    stride = (pitch * ROWS + pitch * ch + 255) // 256 * 256
    out = torch.zeros((d.shape[0], stride), dtype=torch.uint8, device=d.device)
    out[:, : pitch * H].view(-1, H, pitch)[:, :, :W] = d[:, : W * H].view(-1, H, W)
    uv = out[:, pitch * ROWS: pitch * ROWS + pitch * ch].view(-1, ch, pitch)
    uv[:, :, 0: 2 * cw: 2] = d[:, W * H: W * H + cw * ch].view(-1, ch, cw)
    uv[:, :, 1: 2 * cw: 2] = d[:, W * H + cw * ch: W * H + 2 * cw * ch].view(-1, ch, cw)
    return out, stride, pitch


def pitched(d, fmt):
    ch, cw = h2j_b200.chroma_shape(W, H, fmt)
    stride = 3 * PITCH * ROWS
    out = torch.zeros((d.shape[0], stride), dtype=torch.uint8, device=d.device)
    out[:, : PITCH * H].view(-1, H, PITCH)[:, :, :W] = d[:, : W * H].view(-1, H, W)
    for k in (1, 2):
        src = d[:, W * H + (k - 1) * cw * ch: W * H + k * cw * ch].view(-1, ch, cw)
        out[:, k * PITCH * ROWS: k * PITCH * ROWS + PITCH * ch].view(-1, ch, PITCH)[:, :, :cw] = src
    return out, stride


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    result = {"what": f"device-resident frames/s, {N} x {W}x{H} per launch, {a.steps} launches per sample, {a.rounds} alternated rounds",
              "gpu": gpu_identity(), "variants": {}}
    pick = [0, 97, 200, 311, 402, 511]
    for fmt, tag in ((1, "422"), (2, "444")):
        planar = make_frames_torch(N, W, H, dev, seed0=9000 + fmt, chroma_format=fmt)
        d_planar, fb, pstride = planar
        want = {}
        ch, cw = h2j_b200.chroma_shape(W, H, fmt)
        for i in pick:
            f = d_planar[i, :fb].cpu().numpy()
            want[i] = orc.oracle_encode(f[: W * H].reshape(H, W), f[W * H: W * H + cw * ch].reshape(ch, cw),
                                        f[W * H + cw * ch: fb].reshape(ch, cw), chroma_format=fmt)[0]
        sp, sp_stride, sp_pitch = semiplanar(d_planar, fmt)
        sp_name = "nv16" if fmt == 1 else "nv24"
        enc = h2j_b200.Encoder(max_width=W, max_height=H, max_batch=N, n_slots=1, chroma_format=fmt, max_jpeg_bytes=4 * 1024 * 1024)
        st = torch.cuda.Stream(device=dev)
        enc.set_stream(0, st.cuda_stream)

        def sp_submit(prepass):
            def go():
                enc.set_knob("semiplanar_prepass", prepass)
                enc.submit_device_semiplanar(0, sp.data_ptr(), sp_stride, sp_pitch, sp_pitch * ROWS, N, W, H)
            return go

        variants = {f"{tag}_planar": lambda: enc.submit_device(0, d_planar.data_ptr(), pstride, N, W, H),
                    f"{sp_name}_in_place": sp_submit(0), f"{sp_name}_prepass": sp_submit(1)}
        if fmt == 2:
            pt, pt_stride = pitched(d_planar, fmt)
            variants["444_pitched_nvdec_layout"] = lambda: enc.submit_device_pitched(0, pt.data_ptr(), pt_stride, PITCH, PITCH,
                                                                                        PITCH * ROWS, 2 * PITCH * ROWS, N, W, H)
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
                bad = [i for i in pick if int(status[i]) != 0 or enc.read_device(d_out + i * cap, int(sizes[i])) != want[i]]
                parity[k].append(not bad)
        enc.close()
        for k in variants:
            s = samples[k]
            result["variants"][k] = {"frames_per_s_median": round(statistics.median(s)), "min": round(min(s)), "max": round(max(s)),
                                     "kernel_launches_per_batch": launches[k], "parity_6_frames_every_round": all(parity[k])}
        del d_planar, sp, planar
        torch.cuda.empty_cache()
    v = result["variants"]
    result["in_place_over_prepass"] = {n: round(v[f"{n}_in_place"]["frames_per_s_median"] / v[f"{n}_prepass"]["frames_per_s_median"], 3)
                                       for n in ("nv16", "nv24")}
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not all(x["parity_6_frames_every_round"] for x in v.values()):
        sys.exit(1)


if __name__ == "__main__":
    main()
