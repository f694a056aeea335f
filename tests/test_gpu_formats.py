"""GPU suite, row f3: the encoder at 4:2:2 and 4:4:4 (settings.chroma_format) against the oracle's chroma_format modes -- which
tests/test_oracle_vs_reference.py pins live against the libavcodec the reference vendors and tests/golden/golden_frames_fmt.json
pins on the GPU box -- coefficients, histograms, tables and bytes; single pictures, batches with several tiles per CTA, partial
tiles, odd sizes, range conversion."""
import hashlib
import json
import os

import numpy as np
import pytest

from tests.support.layouts import CASES, upload

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("fmt", [1, 2])
def test_frames_match_the_oracle(orc, fmt):
    import h2j_b200

    with h2j_b200.Encoder(max_width=1920, max_height=1088, max_batch=2, n_slots=1, chroma_format=fmt, max_jpeg_bytes=8 * 1024 * 1024) as e:
        for i, (w, h, kind, amp) in enumerate(CASES):
            y, u, v = orc.synth_planes_fmt(w, h, fmt, kind, seed=20 + i, amp=amp)
            want, dbg, coefs = orc.oracle_encode(y, u, v, chroma_format=fmt, want_coefs=True)
            got = e.yuv2jpeg(y, u, v)
            info = e.frame_info(0, 0)
            assert info.mb_var_sum == dbg.mb_var_sum and info.qscale == dbg.qscale, (w, h)
            assert (info.mcu_w, info.mcu_h) == (dbg.mcu_w, dbg.mcu_h)
            got_coefs = e.coefficients(0, 0, coefs.shape[0])
            bad = np.nonzero((got_coefs != coefs).any(axis=1))[0]
            assert bad.size == 0, f"{w}x{h} fmt {fmt}: {bad.size} blocks differ, first {bad[:5]}"
            for t in range(4):
                assert list(info.hist[t]) == list(dbg.hist[t]), f"{w}x{h} fmt {fmt}: histogram {t}"
                assert bytes(info.bits[t]) == bytes(dbg.bits[t])
            assert info.header_bytes == dbg.header_bytes and info.scan_bits == dbg.scan_bits
            assert got == want, f"{w}x{h} {kind} fmt {fmt}"


def test_golden_digests_of_libavcodec_at_422_and_444(orc):
    """against what the libavcodec the reference vendors wrote (tests/golden/make_golden.py formats) -- no oracle in between"""
    import h2j_b200

    d = json.load(open(os.path.join(G, "golden_frames_fmt.json")))
    encs = {}
    try:
        for fr in d["frames"]:
            fmt = fr["chroma_format"]
            if fmt not in encs:
                encs[fmt] = h2j_b200.Encoder(max_width=1920, max_height=1088, max_batch=1, n_slots=1, chroma_format=fmt)
            y, u, v = orc.golden_planes_fmt(fr["w"], fr["h"], fr["seed"], fr["amp"], fmt)
            assert hashlib.sha256(y.tobytes() + u.tobytes() + v.tobytes()).hexdigest() == fr["planes_sha256"], "frame generator drifted"
            j = encs[fmt].yuv2jpeg(y, u, v)
            assert len(j) == fr["size"] and hashlib.sha256(j).hexdigest() == fr["sha256"], fr
    finally:
        for e in encs.values():
            e.close()


@pytest.mark.parametrize("fmt,w,h", [(1, 641, 479), (2, 641, 479), (1, 330, 225), (2, 330, 225), (2, 1918, 1078), (1, 2562, 1442)])
def test_batches_with_several_tiles_per_cta_and_partial_tiles(orc, fmt, w, h):
    import h2j_b200

    n = 6
    planes = [orc.synth_planes_fmt(w, h, fmt, "textured" if s % 3 else "noise", seed=400 + s, amp=12 + 11 * s) for s in range(n)]
    want = [orc.oracle_encode(*p, chroma_format=fmt)[0] for p in planes]
    frames = np.stack([orc.pack_i420(*p) for p in planes])
    assert frames.shape[1] == h2j_b200.frame_bytes(w, h, fmt)
    stride = (frames.shape[1] + 255) // 256 * 256
    d, ptr = upload(frames, stride)
    with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=n, n_slots=1, chroma_format=fmt, max_jpeg_bytes=8 * 1024 * 1024) as e:
        for tpc in (0, 2, 5, 16):
            e.set_knob("fdct_tiles_per_cta", tpc)
            e.submit_device(0, ptr, stride, n, w, h)
            res = e.collect(0)
            assert res.status == [0] * n
            for i in range(n):
                assert res.jpegs[i] == want[i], f"fmt {fmt} {w}x{h}, {tpc} tiles per CTA, frame {i}"
        e.set_knob("fdct_tiles_per_cta", 0)
        assert e.encode_batch(frames, w, h).jpegs == want  # host frames (odd widths: re-pitched on the device first)


def test_range_conversion_fixed_qscale_and_refusals(orc):
    import torch

    import h2j_b200

    w, h = 322, 242
    for fmt in (1, 2):
        y, u, v = orc.synth_planes_fmt(w, h, fmt, "textured", seed=77, amp=70)
        for kw in ({"range_mode": 1}, {"fixed_qscale": 3}, {"fixed_qscale": 1}):
            with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=1, n_slots=1, chroma_format=fmt, max_jpeg_bytes=8 * 1024 * 1024, **kw) as e:
                assert e.yuv2jpeg(y, u, v) == orc.oracle_encode(y, u, v, chroma_format=fmt, **kw)[0], (fmt, kw)
        with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=1, n_slots=1, chroma_format=fmt) as e:
            # planes of another format's size are refused by the binding, NV12 (a 4:2:0 layout) by the library
            y0, u0, v0 = orc.synth_planes(w, h, "textured", seed=1)
            with pytest.raises(h2j_b200.H2JError):
                e.yuv2jpeg(y0, u0, v0)
            dd = torch.zeros(w * h * 2, dtype=torch.uint8, device="cuda")
            with pytest.raises(h2j_b200.H2JError) as ei:
                e.submit_device_nv12(0, dd.data_ptr(), w * h * 2, 384, 384 * h, 1, w, h)
            assert ei.value.status == h2j_b200.ERR_UNSUPPORTED
            with pytest.raises(h2j_b200.H2JError):
                e.convert_pad(y, u, v, 0)


@pytest.mark.parametrize("fmt", [1, 2])
def test_randomised_geometries_and_contents(orc, fmt):
    """sizes and contents drawn at random (seeded): every width / height residue of the MCU grid, sparse and dense blocks"""
    import h2j_b200

    rng = np.random.default_rng(1000 + fmt)
    kinds = ["textured", "noise", "blocks", "const", "binary", "ff"]
    with h2j_b200.Encoder(max_width=400, max_height=300, max_batch=1, n_slots=1, chroma_format=fmt, max_jpeg_bytes=4 * 1024 * 1024) as e:
        for i in range(40):
            w, h = int(rng.integers(2, 400)), int(rng.integers(2, 300))
            kind = kinds[int(rng.integers(0, len(kinds)))]
            y, u, v = orc.synth_planes_fmt(w, h, fmt, kind, seed=int(rng.integers(0, 1 << 30)), amp=int(rng.integers(1, 128)))
            assert e.yuv2jpeg(y, u, v) == orc.oracle_encode(y, u, v, chroma_format=fmt)[0], (fmt, w, h, kind, i)
