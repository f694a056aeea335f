#!/usr/bin/env python
"""Generates the committed golden vectors FROM THE REFERENCE ITSELF (run in the build container, where
/root/reference exists and oracle/_ref has been built by oracle/Makefile):

  golden_frames.json   sha256 / size / DQT of the JPEG the reference's Encoder::yuv2Jpeg writes for
                       integer-generated frames (tests/support/oracle.py::golden_planes)
  ref_img_crops.npz    256x256 crops of the frames the reference decodes from ITS OWN fixtures
                       (test/img/img01.h264, img01.h265) with the JPEG the reference makes of each crop,
                       plus the sha256 of the full-frame JPEGs (== the fixtures test/img/*.jpeg modulo the
                       COM version string of the h265 one, see DESIGN.md)
  fdct_vectors.npz     8x8 blocks and what the libavcodec the reference links (AVDCT, dct_algo auto ->
                       ff_fdct_sse2) makes of them
  ratecontrol.json     (mb_var_sum, qscale) pairs observed from the reference around every qscale threshold
  swscale_lut.npz      libswscale yuv420p -> yuvj420p mapping of all 256 values (luma, chroma)
  golden_frames_fmt.json   the same encoder at 4:2:2 and 4:4:4 (DESIGN.md row f3): sha256 / size of what the libavcodec the
                       reference vendors makes of integer-generated yuvj422p / yuvj444p frames, opened the way the reference
                       opens it (oracle/ref_harness.cpp ref_mjpeg_encode_fmt).  `python make_golden.py formats` writes only this.
  reference_cases.json digests of what the reference makes of the inputs of tests/test_oracle_vs_reference.py (4:2:0 frames,
                       pts / pix_fmt variants, FDCT blocks, libswscale range conversion, 4:2:2 / 4:4:4 frames), so
                       that those tests compare with the reference where it is absent.  `python make_golden.py cases`
                       writes only this.  `python make_golden.py cases-from-oracle` writes it from the oracle instead and
                       says so in "made_with": valid only at a commit whose tests/test_oracle_vs_reference.py passed live
                       against the reference with the same oracle and the same inputs (that run pinned oracle == reference
                       on every encode, FDCT and range case; for the pts / pix_fmt and 4:2:0-entry frames it pinned that the
                       reference's outputs agree with each other, and the digests are the oracle's output of those frames).
"""
import hashlib
import json
import math
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from tests.support import oracle as orc  # noqa: E402

REFIMG = "/root/reference/test/img"

FRAME_CASES = [  # (w, h, seed, amp)
    (16, 16, 1, 10), (2, 2, 2, 60), (17, 17, 3, 30), (33, 47, 4, 8), (64, 64, 5, 100), (131, 77, 6, 20), (322, 242, 7, 12),
    (641, 479, 8, 40), (1280, 720, 9, 6), (1920, 1080, 10, 10), (1918, 1078, 11, 10), (1920, 1080, 12, 50), (3840, 2160, 13, 4),
    (100, 60, 14, 0), (48, 32, 15, 127),
]


def sha(b):
    return hashlib.sha256(b).hexdigest()


FMT_CASES = [  # (w, h, seed, amp)
    (16, 16, 1, 10), (2, 2, 2, 60), (17, 17, 3, 30), (33, 47, 4, 8), (64, 64, 5, 100), (131, 77, 6, 20), (322, 242, 7, 12),
    (641, 479, 8, 40), (1280, 720, 9, 6), (1920, 1080, 10, 10), (1918, 1078, 11, 10), (8, 16, 12, 50), (9, 31, 13, 50), (24, 40, 14, 127),
]


def main_formats():
    R = orc.reference()
    frames = []
    for fmt in (orc.CHROMA_422, orc.CHROMA_444):
        for (w, h, seed, amp) in FMT_CASES:
            y, u, v = orc.golden_planes_fmt(w, h, seed, amp, fmt)
            j = orc.reference_encode_fmt(y, u, v, fmt)
            frames.append({"chroma_format": fmt, "w": w, "h": h, "seed": seed, "amp": amp, "size": len(j), "sha256": sha(j),
                           "planes_sha256": sha(y.tobytes() + u.tobytes() + v.tobytes())})
            print("fmt", fmt, w, h, seed, amp, len(j))
    json.dump({"generator": "tests/golden/make_golden.py formats", "reference": R.ref_version().decode(),
               "pix_fmt": {"1": "yuvj422p", "2": "yuvj444p"}, "frames": frames},
              open(os.path.join(HERE, "golden_frames_fmt.json"), "w"), indent=1)


def main():
    R = orc.reference()
    out = {}
    # ---- frames ---------------------------------------------------------------------------------------
    frames = []
    for (w, h, seed, amp) in FRAME_CASES:
        y, u, v = orc.golden_planes(w, h, seed, amp)
        j = orc.reference_encode(y, u, v)
        assert len(j) < 2 * 1024 * 1024 - 4096
        frames.append({"w": w, "h": h, "seed": seed, "amp": amp, "size": len(j), "sha256": sha(j), "dqt1": j[27],
                       "planes_sha256": sha(y.tobytes() + u.tobytes() + v.tobytes())})
        print("frame", w, h, seed, amp, len(j))
    json.dump({"generator": "tests/golden/make_golden.py", "reference": R.ref_version().decode(), "frames": frames},
              open(os.path.join(HERE, "golden_frames.json"), "w"), indent=1)

    # ---- the reference's own fixtures -------------------------------------------------------------------
    crops = {}
    for name in ("img01.h264", "img01.h265"):
        yb = np.zeros(4096 * 4096, np.uint8); ub = np.zeros(2048 * 2048, np.uint8); vb = np.zeros_like(ub)
        info = np.zeros(8, np.int64)
        assert R.ref_decode_first_frame(os.path.join(REFIMG, name).encode(), yb.ctypes.data, ub.ctypes.data, vb.ctypes.data, yb.size,
                                        info.ctypes.data) == 1
        w, h = int(info[0]), int(info[1]); cw, ch = (w + 1) // 2, (h + 1) // 2
        y = yb[: w * h].reshape(h, w).copy(); u = ub[: cw * ch].reshape(ch, cw).copy(); v = vb[: cw * ch].reshape(ch, cw).copy()
        full = orc.reference_encode(y, u, v)
        shipped = open(os.path.join(REFIMG, name + ".jpeg"), "rb").read()
        # everything after the COM segment must equal the shipped fixture
        assert full[full.find(b"\xff\xdb"):] == shipped[shipped.find(b"\xff\xdb"):], name
        x0, y0 = (w // 3) & ~15, (h // 3) & ~15
        cy = y[y0: y0 + 256, x0: x0 + 256].copy(); cu = u[y0 // 2: y0 // 2 + 128, x0 // 2: x0 // 2 + 128].copy()
        cv = v[y0 // 2: y0 // 2 + 128, x0 // 2: x0 // 2 + 128].copy()
        cj = orc.reference_encode(cy, cu, cv)
        key = name.replace(".", "_")
        crops[key + "_y"], crops[key + "_u"], crops[key + "_v"] = cy, cu, cv
        crops[key + "_jpeg"] = np.frombuffer(cj, np.uint8)
        crops[key + "_full_sha256"] = np.frombuffer(sha(full).encode(), np.uint8)
        crops[key + "_full_dims"] = np.array([w, h, len(full), int(info[2])])
        crops[key + "_shipped_tail_sha256"] = np.frombuffer(sha(shipped[shipped.find(b"\xff\xdb"):]).encode(), np.uint8)
        print(name, w, h, len(full), "crop jpeg", len(cj))
    np.savez_compressed(os.path.join(HERE, "ref_img_crops.npz"), **crops)

    # ---- fdct -----------------------------------------------------------------------------------------
    rng = np.random.default_rng(1234)
    blocks = [rng.integers(0, 256, (384, 64)), rng.integers(100, 140, (64, 64))]
    ext = [np.full(64, 255), np.zeros(64, np.int64)]
    yy, xx = np.mgrid[0:8, 0:8]
    for uu in range(8):
        for vv in range(8):
            b = np.cos((2 * xx + 1) * uu * np.pi / 16) * np.cos((2 * yy + 1) * vv * np.pi / 16)
            ext.append(np.where(b > 0, 255, 0).reshape(64)); ext.append(np.where(b > 0, 0, 255).reshape(64))
    blocks = np.ascontiguousarray(np.concatenate(blocks + [np.array(ext)]).astype(np.int16))
    outb = blocks.copy()
    assert R.ref_fdct(outb.ctypes.data, len(outb)) == 1
    np.savez_compressed(os.path.join(HERE, "fdct_vectors.npz"), blocks=blocks, fdct=outb)

    # ---- rate control: craft luma planes whose mb_var_sum straddles each qscale threshold ----------------
    O = orc.oracle()
    pairs = {}
    rng = np.random.default_rng(99)
    f32 = np.float32

    def lam_of_n(n):
        tex = n * 236.0
        b = math.pow(tex, 0.5) + 1.0
        qd = 236.0 * (n + 1) / b * float(f32(0.8))
        q = float(f32(qd)); q = float(f32((0.0005 + q) / 1.0005))
        return q

    targets = []
    for qs in range(3, 26):  # lambda threshold where update_qscale() steps to qs
        lam_th = math.ceil((qs * 16384 - 8192) / 139)
        n = 1
        while lam_of_n(n) + 0.5 < lam_th:
            n += max(1, n // 200)
        targets.append((qs, n))
    def craft(target, n_mb_w, n_mb_h):
        """Luma plane of constant 8x8 blocks (a b / b a per macroblock): large 16x16 variance, DC-only JPEG."""
        M = n_mb_w * n_mb_h
        def varc(d):
            a_, b_ = 128 - d, 128 + d
            s_ = 128 * (a_ + b_); nrm = 128 * (a_ * a_ + b_ * b_)
            return (nrm - ((s_ * s_) >> 8) + 628) >> 8
        d = 0
        while d < 127 and varc(d + 1) * M <= target:
            d += 1
        k = 0 if d >= 127 else int(round((target - varc(d) * M) / max(1, varc(d + 1) - varc(d))))
        k = max(0, min(M, k))
        ds = np.full(M, d, np.int64); ds[:k] = min(127, d + 1)
        ds = ds.reshape(n_mb_h, n_mb_w)
        pat = np.array([[-1, 1], [1, -1]])
        blocks = 128 + np.kron(ds, pat)                      # (2*mbh, 2*mbw) block values
        return np.kron(blocks, np.ones((8, 8), np.int64)).astype(np.uint8)

    sizes = [(4, 4), (20, 15), (80, 45), (120, 68), (240, 135)]
    for qs, n in targets:
        for dn in (-2, -1, 0, 1, 2):
            var_t = int(((n + dn + 0.5) / 3.5) ** 2)
            mbw, mbh = next(((a_, b_) for (a_, b_) in sizes if var_t / (a_ * b_) < 15000), sizes[-1])
            y = craft(var_t, mbw, mbh)
            h, w = y.shape
            var = int(O.orc_mb_var_sum(y.ctypes.data, w, w, h))
            if var in pairs:
                continue
            c = np.full((h // 2, w // 2), 128, np.uint8)
            j = orc.reference_encode(y, c, c)
            pairs[var] = j[27] // 2
    # plus a spread of random ones
    for t in range(300):
        w = 16 * int(rng.integers(1, 12)); h = 16 * int(rng.integers(1, 12)); amp = int(rng.integers(1, 128))
        y = np.clip(128 + rng.integers(-amp, amp + 1, (h, w)), 0, 255).astype(np.uint8)
        var = int(O.orc_mb_var_sum(y.ctypes.data, w, w, h))
        c = np.full((h // 2, w // 2), 128, np.uint8)
        pairs[var] = orc.reference_encode(y, c, c)[27] // 2
    json.dump({"note": "mb_var_sum -> qscale chosen by the reference (DQT[1] / 2)", "pairs": sorted(pairs.items())},
              open(os.path.join(HERE, "ratecontrol.json"), "w"))
    print("ratecontrol pairs", len(pairs), "qscales", sorted(set(pairs.values())))

    # ---- swscale --------------------------------------------------------------------------------------
    w, h = 32, 16
    lut = np.zeros((2, 256), np.uint8)
    for val in range(256):
        y = np.full((h, w), val, np.uint8); c = np.full((h // 2, w // 2), val, np.uint8)
        oy = np.zeros_like(y); ou = np.zeros_like(c); ov = np.zeros_like(c)
        assert R.ref_sws_limited_to_full(y.ctypes.data, c.ctypes.data, c.ctypes.data, w, h, 2, oy.ctypes.data, ou.ctypes.data, ov.ctypes.data) == 1
        assert (oy == oy[0, 0]).all() and (ou == ou[0, 0]).all() and (ou == ov).all()
        lut[0, val] = oy[0, 0]; lut[1, val] = ou[0, 0]
    np.savez_compressed(os.path.join(HERE, "swscale_lut.npz"), lut=lut)
    print("done")


def main_cases(from_oracle=False):
    from tests import test_oracle_vs_reference as T

    L = orc.oracle()
    if from_oracle:
        made_with = ("the CPU oracle (oracle/mjpeg_oracle.c) at a commit whose tests/test_oracle_vs_reference.py passed live against "
                     "the compiled reference (Lavc58.117.101) on these inputs")
        enc = lambda y, u, v, pts=orc.NOPTS, pix_fmt=0: orc.oracle_encode(y, u, v, pts=pts)[0]  # noqa: E731 (the oracle has no pix_fmt)
        enc_fmt = lambda y, u, v, fmt: orc.oracle_encode(y, u, v, chroma_format=fmt)[0]  # noqa: E731

        def fdct(b):
            for i in range(len(b)):
                L.orc_fdct_sse2(b[i].ctypes.data)

        def rng_conv(w, h, y, u, v, flags):
            return T.oracle_range(orc, w, h, y, u, v)
    else:
        R = orc.reference()
        made_with = "the compiled reference, " + R.ref_version().decode()
        enc, enc_fmt = orc.reference_encode, orc.reference_encode_fmt

        def fdct(b):
            assert R.ref_fdct(b.ctypes.data, len(b)) == 1

        def rng_conv(w, h, y, u, v, flags):
            oy = np.zeros_like(y); ou = np.zeros_like(u); ov = np.zeros_like(v)
            assert R.ref_sws_limited_to_full(y.ctypes.data, u.ctypes.data, v.ctypes.data, w, h, flags, oy.ctypes.data, ou.ctypes.data, ov.ctypes.data) == 1
            return oy, ou, ov

    out = {"generator": "tests/golden/make_golden.py " + ("cases-from-oracle" if from_oracle else "cases"), "made_with": made_with,
           "encode_420": {}, "encode_fmt": {}, "range": {}}
    for (w, h, kind, amp) in T.CASES:
        y, u, v = orc.synth_planes(w, h, kind, seed=w * 7 + h, amp=amp)
        j = enc(y, u, v)
        out["encode_420"][f"{w}x{h}_{kind}_{amp}"] = {"planes_sha256": T.sha(y, u, v), "size": len(j), "sha256": T.sha(j)}
    w, h, kind, seed, amp = T.PTS_FRAME
    y, u, v = orc.synth_planes(w, h, kind, seed=seed, amp=amp)
    variants = {"base": T.sha(enc(y, u, v)), "pix_fmt=12": T.sha(enc(y, u, v, pix_fmt=12))}
    variants.update({f"pts={p}": T.sha(enc(y, u, v, pts=p)) for p in T.PTS})
    out["pts_pix_fmt"] = {"planes_sha256": T.sha(y, u, v), "sha256": variants}
    blocks = T.fdct_blocks()
    coefs = blocks.copy()
    fdct(coefs)
    out["fdct"] = {"blocks_sha256": T.sha(blocks), "fdct_sha256": T.sha(coefs)}
    for (w, h, y, u, v) in T.range_planes():
        out["range"][f"{w}x{h}"] = {"planes_sha256": T.sha(y, u, v)}
        out["range"][f"{w}x{h}"].update({f"flags={f}": T.sha(*rng_conv(w, h, y, u, v, f)) for f in T.RANGE_FLAGS})
    for fmt in (orc.CHROMA_422, orc.CHROMA_444):
        for i, (w, h, kind, amp) in enumerate(T.FMT_CASES):
            y, u, v = orc.synth_planes_fmt(w, h, fmt, kind, seed=50 + i, amp=amp)
            j = enc_fmt(y, u, v, fmt)
            out["encode_fmt"][f"{fmt}_{w}x{h}_{kind}_{amp}"] = {"planes_sha256": T.sha(y, u, v), "size": len(j), "sha256": T.sha(j)}
    w, h, kind, seed = T.FMT0_FRAME
    y, u, v = orc.synth_planes(w, h, kind, seed=seed)
    out["fmt0_entry"] = {"planes_sha256": T.sha(y, u, v), "sha256_fmt_entry": T.sha(enc_fmt(y, u, v, 0)), "sha256_default_entry": T.sha(enc(y, u, v))}
    json.dump(out, open(os.path.join(HERE, "reference_cases.json"), "w"), indent=1)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "formats":
        main_formats()
    elif len(sys.argv) > 1 and sys.argv[1] in ("cases", "cases-from-oracle"):
        main_cases(from_oracle=sys.argv[1] == "cases-from-oracle")
    else:
        main()
        main_formats()
