"""CPU suite: the oracle against the reference on seeded frames, FDCT blocks and range conversions.  Every case is compared
with tests/golden/reference_cases.json, digests of what the reference makes of exactly these inputs (provenance in that
file's "made_with" and in tests/golden/make_golden.py); where the compiled reference is present (oracle/_ref, built from
/root/reference by oracle/Makefile) the same inputs also go through it live.  test_reference_fixtures needs the
reference's decoder and test/img pictures and runs only there."""
import functools
import hashlib
import json
import os

import numpy as np
import pytest

from tests.support import oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_cases.json")

CASES = [(16, 16, "textured", 40), (2, 2, "noise", 100), (3, 5, "noise", 50), (17, 17, "noise", 60), (33, 47, "blocks", 30),
         (64, 64, "binary", 0), (100, 60, "const", 0), (131, 77, "textured", 80), (322, 242, "textured", 40), (641, 479, "noise", 20),
         (1280, 720, "textured", 30), (1918, 1078, "textured", 40), (1920, 1080, "ff", 0)]
PTS = (0, 1, 50, 5000, 100000, -5)
PTS_FRAME = (320, 240, "noise", 5, 60)  # w, h, kind, seed, amp
FDCT_SEED, FDCT_BLOCKS = 5, 4096
RANGE_SEED, RANGE_SIZES, RANGE_FLAGS = 6, [(64, 48), (33, 17), (258, 130)], (2, 4, 0x10)
FMT_CASES = [(64, 48, "textured", 40), (16, 16, "noise", 100), (17, 17, "noise", 60), (33, 47, "blocks", 30), (131, 77, "textured", 80),
             (322, 242, "textured", 40), (641, 479, "noise", 20), (8, 16, "noise", 50), (9, 16, "noise", 50), (24, 40, "textured", 30),
             (1280, 720, "textured", 30), (2, 2, "noise", 100), (25, 9, "binary", 0), (1918, 1078, "textured", 25)]
FMT0_FRAME = (322, 242, "textured", 3)  # w, h, kind, seed


def sha(*parts):
    h = hashlib.sha256()
    for p in parts:
        h.update(p if isinstance(p, bytes) else np.ascontiguousarray(p).tobytes())
    return h.hexdigest()


@functools.lru_cache(maxsize=None)
def golden():
    return json.load(open(GOLDEN))


def fdct_blocks():
    rng = np.random.default_rng(FDCT_SEED)
    return np.ascontiguousarray(rng.integers(0, 256, (FDCT_BLOCKS, 64)).astype(np.int16))


def range_planes():
    """(w, h, y, u, v) of every RANGE_SIZES entry, drawn in order from one generator"""
    rng = np.random.default_rng(RANGE_SEED)
    out = []
    for (w, h) in RANGE_SIZES:
        cw, ch = (w + 1) // 2, (h + 1) // 2
        y = rng.integers(0, 256, (h, w)).astype(np.uint8); u = rng.integers(0, 256, (ch, cw)).astype(np.uint8); v = rng.integers(0, 256, (ch, cw)).astype(np.uint8)
        out.append((w, h, y, u, v))
    return out


def oracle_range(orc, w, h, y, u, v):
    cw, ch = (w + 1) // 2, (h + 1) // 2
    my = np.zeros_like(y); mu = np.zeros_like(u); mv = np.zeros_like(v)
    lib = orc.oracle()
    lib.orc_range_luma(y.ctypes.data, w, my.ctypes.data, w, w, h)
    lib.orc_range_chroma(u.ctypes.data, cw, mu.ctypes.data, cw, cw, ch)
    lib.orc_range_chroma(v.ctypes.data, cw, mv.ctypes.data, cw, cw, ch)
    return my, mu, mv


@pytest.mark.parametrize("w,h,kind,amp", CASES)
def test_oracle_equals_reference(orc, w, h, kind, amp):
    y, u, v = orc.synth_planes(w, h, kind, seed=w * 7 + h, amp=amp)
    rec = golden()["encode_420"][f"{w}x{h}_{kind}_{amp}"]
    assert sha(y, u, v) == rec["planes_sha256"], "frame generator drifted"
    got, _, _ = orc.oracle_encode(y, u, v)
    assert len(got) == rec["size"] and sha(got) == rec["sha256"]
    if orc.have_reference():
        assert got == orc.reference_encode(y, u, v)


def test_reference_ignores_pts_and_pix_fmt(orc):
    w, h, kind, seed, amp = PTS_FRAME
    y, u, v = orc.synth_planes(w, h, kind, seed=seed, amp=amp)
    rec = golden()["pts_pix_fmt"]
    assert sha(y, u, v) == rec["planes_sha256"], "frame generator drifted"
    # what the reference made of the frame with no pts, each pts and a yuvj420p-tagged frame: the same bytes every time
    assert set(rec["sha256"]) == {"base", "pix_fmt=12"} | {f"pts={p}" for p in PTS} and len(set(rec["sha256"].values())) == 1
    assert sha(orc.oracle_encode(y, u, v)[0]) == rec["sha256"]["base"]
    for pts in PTS:
        assert sha(orc.oracle_encode(y, u, v, pts=pts)[0]) == rec["sha256"][f"pts={pts}"]
    if orc.have_reference():
        base = orc.reference_encode(y, u, v)
        assert sha(base) == rec["sha256"]["base"]
        for pts in PTS:
            assert orc.reference_encode(y, u, v, pts=pts) == base
        assert orc.reference_encode(y, u, v, pix_fmt=12) == base  # AV_PIX_FMT_YUVJ420P frame: same bytes


@pytest.mark.skipif(not O.have_reference(), reason="oracle/_ref not built (needs /root/reference)")
@pytest.mark.skipif(not os.path.exists("/root/reference/test/img/img01.h264"), reason="reference fixtures not present")
@pytest.mark.parametrize("name", ["img01.h264", "img01.h265"])
def test_reference_fixtures(orc, name, tmp_path):
    R = orc.reference()
    yb = np.zeros(4096 * 4096, np.uint8); ub = np.zeros(2048 * 2048, np.uint8); vb = np.zeros_like(ub)
    info = np.zeros(8, np.int64)
    path = "/root/reference/test/img/" + name
    assert R.ref_decode_first_frame(path.encode(), yb.ctypes.data, ub.ctypes.data, vb.ctypes.data, yb.size, info.ctypes.data) == 1
    w, h = int(info[0]), int(info[1]); cw, ch = (w + 1) // 2, (h + 1) // 2
    y = yb[: w * h].reshape(h, w).copy(); u = ub[: cw * ch].reshape(ch, cw).copy(); v = vb[: cw * ch].reshape(ch, cw).copy()
    got, _, _ = orc.oracle_encode(y, u, v)
    # the whole reference path, file to file
    out = str(tmp_path / "o.jpeg")
    assert R.ref_h265_to_jpeg(path.encode(), out.encode(), 1) == 1
    assert got == open(out, "rb").read()
    shipped = open(path + ".jpeg", "rb").read()
    # the shipped h265 fixture was produced by another libavcodec build (COM says Lavc58.91.100): equal past COM
    assert got[got.find(b"\xff\xdb"):] == shipped[shipped.find(b"\xff\xdb"):]
    if name == "img01.h264":
        assert got == shipped


def test_fdct_matches_libavcodec(orc):
    blocks = fdct_blocks()
    rec = golden()["fdct"]
    assert sha(blocks) == rec["blocks_sha256"], "block generator drifted"
    lib = orc.oracle()
    got = blocks.copy()
    for i in range(len(got)):
        lib.orc_fdct_sse2(got[i].ctypes.data)
    assert sha(got) == rec["fdct_sha256"]
    if orc.have_reference():
        want = blocks.copy()
        assert orc.reference().ref_fdct(want.ctypes.data, len(want)) == 1
        assert (got == want).all()


def test_range_conversion_matches_libswscale(orc):
    rec = golden()["range"]
    for (w, h, y, u, v) in range_planes():
        assert sha(y, u, v) == rec[f"{w}x{h}"]["planes_sha256"], "plane generator drifted"
        my, mu, mv = oracle_range(orc, w, h, y, u, v)
        for flags in RANGE_FLAGS:
            assert sha(my, mu, mv) == rec[f"{w}x{h}"][f"flags={flags}"], (w, h, flags)
            if orc.have_reference():
                oy = np.zeros_like(y); ou = np.zeros_like(u); ov = np.zeros_like(v)
                assert orc.reference().ref_sws_limited_to_full(y.ctypes.data, u.ctypes.data, v.ctypes.data, w, h, flags, oy.ctypes.data, ou.ctypes.data, ov.ctypes.data) == 1
                assert (my == oy).all() and (mu == ou).all() and (mv == ov).all()


@pytest.mark.parametrize("fmt", [1, 2])
def test_oracle_matches_libavcodec_at_422_and_444(orc, fmt):
    """Row f3: libavcodec's mjpeg encoder opened as reference src/Encoder.cpp:158-204 opens it but as yuvj422p / yuvj444p
    (the reference itself hard-codes yuvj420p, :162) against the oracle's chroma_format modes, byte for byte."""
    recs = golden()["encode_fmt"]
    for i, (w, h, kind, amp) in enumerate(FMT_CASES):
        y, u, v = orc.synth_planes_fmt(w, h, fmt, kind, seed=50 + i, amp=amp)
        rec = recs[f"{fmt}_{w}x{h}_{kind}_{amp}"]
        assert sha(y, u, v) == rec["planes_sha256"], ("frame generator drifted", fmt, w, h, kind)
        got = orc.oracle_encode(y, u, v, chroma_format=fmt)[0]
        assert len(got) == rec["size"] and sha(got) == rec["sha256"], (fmt, w, h, kind)
        if orc.have_reference():
            assert got == orc.reference_encode_fmt(y, u, v, fmt), (fmt, w, h, kind)
    # 4:2:0 through the same entry is the reference's own path
    w, h, kind, seed = FMT0_FRAME
    y, u, v = orc.synth_planes(w, h, kind, seed=seed)
    rec = golden()["fmt0_entry"]
    assert sha(y, u, v) == rec["planes_sha256"], "frame generator drifted"
    assert rec["sha256_fmt_entry"] == rec["sha256_default_entry"] == sha(orc.oracle_encode(y, u, v)[0])
    if orc.have_reference():
        assert orc.reference_encode_fmt(y, u, v, 0) == orc.reference_encode(y, u, v)
        assert sha(orc.reference_encode(y, u, v)) == rec["sha256_default_entry"]
