#!/usr/bin/env python
"""Device-resident throughput of list batches (h2j_submit_device_list, DESIGN.md row (f)(6)), frames/s:

  (a) uniform_submit_device / uniform_list: 512 x 1080p through h2j_submit_device, and the same frames through the list
      entry point (what the descriptor table costs on uniform input)
  (b) alternating_list / alternating_two_uniform: 512 frames alternating 1920x1080 / 1280x720 in one list submit, against
      the same frames as two uniform submits (256 x 1080p, then 256 x 720p) back to back on one slot
  (c) alternating_batch1: the same 512 frames one submit each (what a batch scope that seals on every size change did)
  (d) skewed_list / skewed_two_uniform: one 3840x2160 frame and 255 at 1280x720 in one list submit (every frame's grid is
      the 4K frame's: what the empty CTAs cost), against the 4K frame and the 255 small ones as two uniform submits

Every variant is warmed up; then rounds of one timed sample per variant (STEPS repetitions of the workload, submit +
collect_device, CUDA events on the slot's stream) alternate the variants, and the line reports the median and the spread
(min, max) of frames/s over the rounds.  After every timed sample up to six frames of its last launch are compared with the
oracle's JPEG.  The working set (1.6 GB of 1080p frames) is far larger than L2.  Prints one JSON line (and writes it to
--out).  Run on the GPU box: python tools/mixed_batch_probe.py --out FILE"""
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

N = 512


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


class Pool:
    """n tight I420 frames of one size in one device buffer"""

    def __init__(self, n, w, h, dev, seed0):
        self.w, self.h = w, h
        self.d, self.fb, self.stride = make_frames_torch(n, w, h, dev, seed0=seed0)
        self.want = {}

    def ptr(self, i):
        return self.d.data_ptr() + i * self.stride

    def desc(self, i):
        w, h = self.w, self.h
        cw, ch = (w + 1) // 2, (h + 1) // 2
        return h2j_b200.FrameDesc(self.ptr(i), w, h, w, cw, w * h, w * h + cw * ch)

    def oracle(self, i):
        if i not in self.want:
            w, h = self.w, self.h
            cw, ch = (w + 1) // 2, (h + 1) // 2
            f = self.d[i, : self.fb].cpu().numpy()
            self.want[i] = orc.oracle_encode(f[: w * h].reshape(h, w), f[w * h: w * h + cw * ch].reshape(ch, cw),
                                             f[w * h + cw * ch:].reshape(ch, cw))[0]
        return self.want[i]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    p1080 = Pool(N, 1920, 1080, dev, 7100)
    p720 = Pool(N, 1280, 720, dev, 7200)
    p4k = Pool(1, 3840, 2160, dev, 7300)
    enc = h2j_b200.Encoder(max_width=3840, max_height=2160, max_batch=N, n_slots=1, max_jpeg_bytes=4 * 1024 * 1024)
    st = torch.cuda.Stream(device=dev)
    enc.set_stream(0, st.cuda_stream)

    # a workload: a list of launches, each (submit function, [(pool, index) of frame k of the launch])
    def uniform(pool, idx):
        return (lambda: enc.submit_device(0, pool.ptr(idx[0]), pool.stride, len(idx), pool.w, pool.h), [(pool, i) for i in idx])

    def listed(frames):
        descs = [p.desc(i) for p, i in frames]
        return (lambda: enc.submit_device_list(0, h2j_b200.LAYOUT_PLANAR, descs), frames)

    alternating = [(p1080, i // 2) if i % 2 == 0 else (p720, i // 2) for i in range(N)]
    skewed = [(p4k, 0)] + [(p720, i) for i in range(255)]
    workloads = {
        "a_uniform_submit_device": [uniform(p1080, list(range(N)))],
        "a_uniform_list": [listed([(p1080, i) for i in range(N)])],
        "b_alternating_list": [listed(alternating)],
        "b_alternating_two_uniform": [uniform(p1080, list(range(N // 2))), uniform(p720, list(range(N // 2)))],
        "c_alternating_batch1": [uniform(p, [i]) for p, i in alternating],
        "d_skewed_list": [listed(skewed)],
        "d_skewed_two_uniform": [uniform(p4k, [0]), uniform(p720, list(range(255)))],
    }
    n_frames = {k: sum(len(f) for _, f in w) for k, w in workloads.items()}

    def run(w):
        for go, _ in w:
            go()
            out = enc.collect_device(0)
        return out

    def parity(w, out):
        d_out, cap, sizes, status = out
        frames = w[-1][1]
        ks = sorted({0, len(frames) - 1} | set(range(0, len(frames), max(1, len(frames) // 4))))[:6]
        return all(int(status[k]) == 0 and enc.read_device(d_out + k * cap, int(sizes[k])) == frames[k][0].oracle(frames[k][1]) for k in ks)

    torch.cuda.synchronize()
    launches = {}
    for k, w in workloads.items():  # warm-up, and the kernel launches one repetition takes
        before = enc.kernel_launches
        run(w)
        launches[k] = enc.kernel_launches - before
    samples = {k: [] for k in workloads}
    ok = {k: [] for k in workloads}
    for _ in range(a.rounds):
        for k, w in workloads.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(a.steps):
                out = run(w)
            e1.record(st)
            e1.synchronize()
            samples[k].append(n_frames[k] * a.steps / (e0.elapsed_time(e1) / 1000.0))
            ok[k].append(parity(w, out))
    enc.close()
    result = {"what": f"device-resident frames/s, {a.steps} repetitions of each workload per sample, {a.rounds} alternated rounds",
              "gpu": gpu_identity(), "variants": {}}
    for k in workloads:
        s = samples[k]
        result["variants"][k] = {"frames": n_frames[k], "frames_per_s_median": round(statistics.median(s)), "min": round(min(s)),
                                 "max": round(max(s)), "kernel_launches": launches[k], "parity_every_round": all(ok[k])}
    v = result["variants"]
    med = {k: x["frames_per_s_median"] for k, x in v.items()}
    result["ratios"] = {
        "a_list_over_submit_device": round(med["a_uniform_list"] / med["a_uniform_submit_device"], 3),
        "b_list_over_two_uniform": round(med["b_alternating_list"] / med["b_alternating_two_uniform"], 3),
        "c_list_over_batch1": round(med["b_alternating_list"] / med["c_alternating_batch1"], 3),
        "d_list_over_two_uniform": round(med["d_skewed_list"] / med["d_skewed_two_uniform"], 3),
    }
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not all(x["parity_every_round"] for x in v.values()):
        sys.exit(1)


if __name__ == "__main__":
    main()
