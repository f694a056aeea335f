"""GPU suite: high-bit-depth input (DESIGN.md row (f)(5)) -- P010 / P216-family semi-planar and 16-bit planar device frames
(h2j_submit_device_semiplanar16 / h2j_submit_device_pitched16), single 16-bit pictures from the host (h2j_encode_frame16)
and the host class's yuv420p10le / yuv420p12le pictures.

Every 16-bit frame is made from 8-bit planes p as word = (p << (d - 8)) | noise below | garbage above bit d (d < 16), so the
expected JPEG is always the oracle's JPEG of p: the low noise and the high garbage must never reach the picture.  Padding
words between rows and planes are 0xA5A5.  A device submit must take exactly one launch more than the pipeline."""
import ctypes as C
import os

import numpy as np
import pytest

from tests.support.layouts import BIG_JPEG, CASES, align, pipeline_launches, place, run, upload

pytestmark = pytest.mark.gpu

PAD16 = 0xA5A5
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST_SO = os.path.join(ROOT, "h264-h265-to-jpeg_b200", "lib", "libh2j_host.so")
YUV420P10LE, YUV420P12LE, YUV420P10BE = 64, 125, 63  # AVPixelFormat of libavutil 56


def widen(p, d, rng):
    """8-bit plane -> 16-bit words holding p in bits [d - 8, d), random bits below and (d < 16) random bits above"""
    w = (p.astype(np.uint16) << (d - 8)) | rng.integers(0, 1 << (d - 8), p.shape, dtype=np.uint16)
    if d < 16:
        w |= rng.integers(0, 1 << (16 - d), p.shape, dtype=np.uint16) << d
    return w


def sp_layout(w, h, fmt, layout):
    """(pitch, uv_off, size, base shift) in bytes"""
    import h2j_b200

    ch, cw = h2j_b200.chroma_shape(w, h, fmt)
    row = 2 * max(w, 2 * cw)
    if layout == "decoder":  # pitch rounded to 256, pair plane behind luma rows padded to a multiple of 16
        pitch = align(row, 256)
        uv_off, shift = pitch * align(h, 16), 0
    elif layout == "tight":
        pitch, uv_off, shift = row, row * h, 0
    else:  # base and pitch 2 (mod 16)
        pitch = align(row, 16) + 2
        uv_off, shift = pitch * h, 2
    return pitch, uv_off, uv_off + pitch * ch, shift


def pl_layouts(w, h, fmt):
    """name -> (y_pitch, c_pitch, u_off, v_off, size, base shift), bytes"""
    import h2j_b200

    ch, cw = h2j_b200.chroma_shape(w, h, fmt)
    out = {"tight": (2 * w, 2 * cw, 2 * w * h, 2 * w * h + 2 * cw * ch, 2 * (w * h + 2 * cw * ch), 0)}
    p, sh = align(2 * w, 256), align(h, 16)  # a decoder's 16-bit surface: one pitch, planes at multiples of pitch * surface height
    out["decoder"] = (p, p, p * sh, 2 * p * sh, 2 * p * sh + p * ch, 0)
    out["yv12"] = (2 * w, 2 * cw, 2 * (w * h + cw * ch), 2 * w * h, 2 * (w * h + 2 * cw * ch), 0)  # V in front of U
    yp, cp = align(2 * w, 16) + 2, align(2 * cw, 16) + 6
    out["unaligned"] = (yp, cp, yp * h + 4, yp * h + 4 + cp * ch + 8, yp * h + 12 + 2 * cp * ch, 2)
    return out


# ---- semi-planar, every chroma format ----------------------------------------------------------------------------

@pytest.mark.parametrize("layout", ["decoder", "tight", "unaligned"])
@pytest.mark.parametrize("depth", [16, 10])
@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_semiplanar16_matches_oracle(orc, fmt, depth, layout):
    import h2j_b200

    rng = np.random.default_rng(1000 * fmt + depth)
    with h2j_b200.Encoder(max_width=1920, max_height=1088, max_batch=2, n_slots=1, chroma_format=fmt, max_jpeg_bytes=BIG_JPEG) as e:
        P = pipeline_launches(e)
        for i, (w, h, kind, amp) in enumerate(CASES):
            pitch, uv_off, size, shift = sp_layout(w, h, fmt, layout)
            stride = align(size, 256)
            planes = [orc.synth_planes_fmt(w, h, fmt, kind, seed=300 + 2 * i + s, amp=amp) for s in range(2)]
            want = [orc.oracle_encode(*p, chroma_format=fmt)[0] for p in planes]
            d, ptr = upload([place(*(widen(x, depth, rng) for x in p), pitch, pitch, uv_off, size=size) for p in planes], stride, shift)
            got, launches = run(e, lambda: e.submit_device_semiplanar16(0, ptr, stride, pitch, uv_off, depth, 2, w, h), 2)
            for k in range(2):
                assert got[k] == want[k], f"fmt {fmt} depth {depth} {layout} {w}x{h} frame {k}: JPEG differs from the oracle's"
            assert launches == P + 1, f"fmt {fmt} {layout} {w}x{h}: {launches} launches, expected {P + 1}"


# ---- planar at any layout ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_pitched16_matches_oracle(orc, fmt):
    import h2j_b200

    rng = np.random.default_rng(77 + fmt)
    for (w, h) in ((1920, 1080), (641, 479), (33, 17), (2, 2)):
        n = 2
        planes = [orc.synth_planes_fmt(w, h, fmt, "textured", seed=700 + s, amp=30 + 20 * s) for s in range(n)]
        want = [orc.oracle_encode(*p, chroma_format=fmt)[0] for p in planes]
        # (pipeline_launches submits a 16 x 16 frame)
        with h2j_b200.Encoder(max_width=max(w, 16), max_height=max(h, 16), max_batch=n, n_slots=1, chroma_format=fmt,
                              max_jpeg_bytes=BIG_JPEG) as e:
            P = pipeline_launches(e)
            for depth in (9, 10, 12, 16):
                for name, (yp, cp, uo, vo, size, shift) in pl_layouts(w, h, fmt).items():
                    stride = align(size, 256)
                    d, ptr = upload([place(*(widen(x, depth, rng) for x in p), yp, cp, uo, vo, size) for p in planes], stride, shift)
                    got, launches = run(e, lambda: e.submit_device_pitched16(0, ptr, stride, yp, cp, uo, vo, depth, n, w, h), n)
                    assert got == want, f"fmt {fmt} depth {depth} {w}x{h} {name}"
                    assert launches == P + 1, f"fmt {fmt} {w}x{h} {name}: {launches} launches"


# ---- P010 at depth 16 is the NV12 frame of its high bytes ------------------------------------------------------

def test_p010_equals_nv12_of_high_bytes(orc):
    import h2j_b200

    rng = np.random.default_rng(5)
    for (w, h) in ((1920, 1080), (330, 241), (17, 9)):
        ch = (h + 1) // 2
        planes = [orc.synth_planes(w, h, "textured", seed=90 + s) for s in range(2)]
        wide = [[widen(x, 16, rng) for x in p] for p in planes]
        high = [[(x >> 8).astype(np.uint8) for x in p] for p in wide]
        pitch, uv_off, size, _ = sp_layout(w, h, 0, "decoder")
        stride = align(size, 256)
        d16, p16 = upload([place(*p, pitch, pitch, uv_off, size=size) for p in wide], stride)
        npitch, nuv = pitch // 2, pitch // 2 * align(h, 16)
        nsize = nuv + npitch * ch
        d8, p8 = upload([place(*p, npitch, npitch, nuv, size=nsize) for p in high], align(nsize, 256))
        with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=2, n_slots=1) as e:
            got, _ = run(e, lambda: e.submit_device_semiplanar16(0, p16, stride, pitch, uv_off, 16, 2, w, h), 2)
            for prepass in (0, 1):  # both paths of the 8-bit entry
                e.set_knob("semiplanar_prepass", prepass)
                ref, _ = run(e, lambda: e.submit_device_nv12(0, p8, align(nsize, 256), npitch, nuv, 2, w, h), 2)
                assert got == ref, (w, h, prepass)
        assert got == [orc.oracle_encode(*p)[0] for p in planes], (w, h)


# ---- batches, tiles per CTA, the grid's row dimension ----------------------------------------------------------

@pytest.mark.parametrize("fmt,w,h,n", [(0, 641, 479, 5), (1, 641, 479, 5), (2, 641, 479, 5), (0, 7680, 4320, 1), (0, 17, 4098, 2),
                                       (2, 17, 4098, 2)])
def test_batches_across_tiles(orc, fmt, w, h, n):
    import h2j_b200

    rng = np.random.default_rng(w + h + fmt)
    planes = [orc.synth_planes_fmt(w, h, fmt, "textured" if s % 3 else "noise", seed=500 + s, amp=12 + 11 * s) for s in range(n)]
    want = [orc.oracle_encode(*p, chroma_format=fmt)[0] for p in planes]
    pitch, uv_off, size, _ = sp_layout(w, h, fmt, "decoder")
    stride = align(size, 256)
    d, ptr = upload([place(*(widen(x, 10, rng) for x in p), pitch, pitch, uv_off, size=size) for p in planes], stride)
    with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=n, n_slots=1, chroma_format=fmt, max_jpeg_bytes=64 << 20) as e:
        for tpc in (0, 2, 16):
            e.set_knob("fdct_tiles_per_cta", tpc)
            got, _ = run(e, lambda: e.submit_device_semiplanar16(0, ptr, stride, pitch, uv_off, 10, n, w, h), n)
            for i in range(n):
                assert got[i] == want[i], f"fmt {fmt} {w}x{h}, {tpc} tiles per CTA, frame {i}"


# ---- range conversion and fixed qscale -----------------------------------------------------------------------

@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_range_conversion_and_fixed_qscale(orc, fmt):
    import h2j_b200

    rng = np.random.default_rng(9)
    w, h = 322, 242
    y, u, v = orc.synth_planes_fmt(w, h, fmt, "textured", seed=77, amp=70)
    pitch, uv_off, size, _ = sp_layout(w, h, fmt, "tight")
    ds, ps = upload([place(*(widen(x, 10, rng) for x in (y, u, v)), pitch, pitch, uv_off, size=size)], size)
    yp, cp, uo, vo, psize, _ = pl_layouts(w, h, fmt)["decoder"]
    dp, pp = upload([place(*(widen(x, 12, rng) for x in (y, u, v)), yp, cp, uo, vo, psize)], align(psize, 256))
    for kw in ({"range_mode": 1}, {"fixed_qscale": 1}, {"fixed_qscale": 31}):
        want = orc.oracle_encode(y, u, v, chroma_format=fmt, **kw)[0]
        with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=1, n_slots=1, chroma_format=fmt, max_jpeg_bytes=BIG_JPEG, **kw) as e:
            got, _ = run(e, lambda: e.submit_device_semiplanar16(0, ps, size, pitch, uv_off, 10, 1, w, h), 1)
            assert got[0] == want, (fmt, kw, "semi-planar")
            got, _ = run(e, lambda: e.submit_device_pitched16(0, pp, align(psize, 256), yp, cp, uo, vo, 12, 1, w, h), 1)
            assert got[0] == want, (fmt, kw, "planar")
            wide = [widen(x, 16, rng) for x in (y, u, v)]
            assert e.yuv2jpeg16(*wide, 16) == want, (fmt, kw, "host")


# ---- single pictures from the host -----------------------------------------------------------------------------

def strided(a, pad):
    """a copy of `a` inside a wider array: rows `pad` words longer"""
    big = np.full((a.shape[0], a.shape[1] + pad), PAD16, np.uint16)
    big[:, : a.shape[1]] = a
    return big[:, : a.shape[1]]


def test_encode_frame16_strided_and_pinned(orc):
    import h2j_b200

    rng = np.random.default_rng(3)
    with h2j_b200.Encoder(max_width=1920, max_height=1088, max_batch=1, n_slots=1, max_jpeg_bytes=BIG_JPEG) as e:
        for (w, h) in ((1920, 1080), (333, 241), (17, 9), (2, 2)):
            y, u, v = orc.synth_planes(w, h, "textured", seed=w, amp=35)
            want = orc.oracle_encode(y, u, v)[0]
            for depth in (10, 12, 16):
                wide = [widen(x, depth, rng) for x in (y, u, v)]
                assert e.yuv2jpeg16(*wide, depth) == want, (w, h, depth, "tight")
                assert e.yuv2jpeg16(*(strided(x, 3 + k) for k, x in enumerate(wide)), depth) == want, (w, h, depth, "strided")
                bufs = [h2j_b200.PinnedBuffer(x.nbytes) for x in wide]
                pinned = [b.array.view(np.uint16).reshape(x.shape) for b, x in zip(bufs, wide)]
                for dst, x in zip(pinned, wide):
                    dst[:] = x
                assert e.yuv2jpeg16(*pinned, depth) == want, (w, h, depth, "pinned")
                del pinned
                for b in bufs:
                    b.free()
        # the 8-bit entry is unchanged after the 16-bit one
        y, u, v = orc.synth_planes(322, 242, "textured", seed=1)
        assert e.yuv2jpeg(y, u, v) == orc.oracle_encode(y, u, v)[0]


def host_lib():
    assert os.path.exists(HOST_SO), "libh2j_host.so missing: run __graft_entry__.build()"
    lib = C.CDLL(HOST_SO)
    lib.h2j_host_yuv2jpeg_file.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_char_p]
    lib.h2j_host_batch_end.argtypes = [C.POINTER(C.c_int)]
    return lib


def write16(lib, planes, fmt, path):
    y, u, v = planes
    h, w = y.shape
    return lib.h2j_host_yuv2jpeg_file(y.ctypes.data, y.strides[0], u.ctypes.data, u.strides[0], v.ctypes.data, v.strides[0], w, h, fmt,
                                      str(path).encode())


def test_host_class_main10_and_main12(orc, tmp_path):
    lib = host_lib()
    rng = np.random.default_rng(11)
    for i, (w, h, fmt, depth) in enumerate(((1920, 1080, YUV420P10LE, 10), (333, 241, YUV420P12LE, 12), (64, 64, YUV420P10LE, 10))):
        y, u, v = orc.synth_planes(w, h, "textured", seed=40 + i, amp=30)
        wide = [strided(widen(x, depth, rng), 8) for x in (y, u, v)]  # AVFrame-like linesizes
        out = tmp_path / f"m_{i}.jpeg"
        assert write16(lib, wide, fmt, out) == 1
        assert out.read_bytes() == orc.oracle_encode(y, u, v)[0], (w, h, fmt)
    # big-endian 10-bit is still refused, and no file is written
    y, u, v = orc.synth_planes(64, 64, "textured", seed=1)
    out = tmp_path / "be.jpeg"
    assert write16(lib, [widen(x, 10, rng) for x in (y, u, v)], YUV420P10BE, out) == 0
    assert not out.exists()


def test_host_class_high_depth_inside_a_batch_scope(orc, tmp_path):
    lib = host_lib()
    rng = np.random.default_rng(12)
    assert lib.h2j_host_batch_begin(4) == 0
    try:
        y, u, v = orc.synth_planes(322, 242, "textured", seed=8, amp=30)
        out = tmp_path / "scope.jpeg"
        assert write16(lib, [widen(x, 10, rng) for x in (y, u, v)], YUV420P10LE, out) == 1
        assert out.read_bytes() == orc.oracle_encode(y, u, v)[0]  # written before yuv2Jpeg returned
    finally:
        failed = C.c_int(-1)
        assert lib.h2j_host_batch_end(C.byref(failed)) == 0 and failed.value == 0
