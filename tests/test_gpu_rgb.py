"""GPU suite: RGB frames (h2j_submit_device_rgb, h2j_encode_frame_rgb).  Every JPEG must be byte-identical to the oracle's
JPEG of the planar frame C(frame) (tests/support/rgb.py) with range_mode 0, and the planes the pipeline read
(h2j_debug_frame_planes) must equal C(frame) bit for bit.  Frames sit in their own allocations surrounded by 0xA5 padding,
pitch and plane gaps are 0xA5 too, and X bytes are random: a byte outside the picture that reached it would change the
planes."""
import ctypes as C
import random

import numpy as np
import pytest

from tests.support import rgb as R
from tests.support.downscale import downscale_planar
from tests.support.layouts import CASES, Frames, align, desc, encoder, pipeline_launches, place, planar, semiplanar, upload

pytestmark = pytest.mark.gpu

GEOMETRIES = CASES + [(17, 4098, "textured", 40)]
MAX_W, MAX_H = 1920, 4098

_pictures = {}


def picture(orc, w, h, kind="textured", amp=40, seed=0):
    """an (H, W, 3) R, G, B picture: three synthetic planes of the kind"""
    key = (w, h, kind, amp, seed)
    if key not in _pictures:
        _pictures[key] = np.stack([orc.synth_planes(w, h, kind, seed=seed + 17 * k, amp=amp)[0] for k in range(3)], -1)
    return _pictures[key]


def want_jpeg(orc, rgb, cf, **kw):
    return orc.oracle_encode(*R.to_planar(rgb, R.RGB24, cf), chroma_format=cf, **kw)[0]


def odd_pitch(n, j):
    return n + 1 + (n % 2) + 2 * j


def layouts(fr, frame, fmt, i):
    """(name, desc) of one frame at every layout the suite covers"""
    h, w = (frame.shape[1:] if fmt == R.PLANAR else frame.shape[:2])
    row = R.BYTES_PER_PIXEL[fmt] * w
    return [
        ("tight", R.place_rgb(fr, frame, fmt)),
        ("decoder", R.place_rgb(fr, frame, fmt, align(row, 256), gap=align(h, 16) - h + 16)),
        ("shifted", R.place_rgb(fr, frame, fmt, odd_pitch(row, i % 3), shift=1 + i % 15, gap=i % 3)),
    ]


@pytest.mark.parametrize("cf", [0, 1, 2])
def test_every_format_geometry_and_layout(orc, cf):
    """per format and layout one list of every size (the list form of the pipeline), every frame against the oracle"""
    import torch

    pics = [picture(orc, w, h, kind, amp, seed=100 + i) for i, (w, h, kind, amp) in enumerate(GEOMETRIES)]
    want = [want_jpeg(orc, p, cf) for p in pics]
    with encoder(cf, len(pics), max_width=MAX_W, max_height=MAX_H) as e:
        for fmt in R.FORMATS:
            fr = Frames()
            per_layout = {}
            for i, p in enumerate(pics):
                for name, d in layouts(fr, R.as_format(p, fmt, seed=i), fmt, i):
                    per_layout.setdefault(name, []).append(d)
            torch.cuda.synchronize()
            for name, descs in per_layout.items():
                e.submit_device_rgb(0, fmt, descs)
                got = e.collect(0).jpegs
                for (w, h, _, _), g, wnt in zip(GEOMETRIES, got, want):
                    assert g == wnt, f"{w}x{h} {R.NAMES[fmt]} chroma {cf} {name}"


@pytest.mark.parametrize("cf", [0, 1, 2])
def test_uniform_list_runs_the_batch_form(orc, cf):
    """frames of one size at their own addresses: the batch form, whose frame info and coefficients match the oracle's,
    one launch more than the pipeline"""
    import torch

    w, h, n = 1283, 723, 4
    pics = [picture(orc, w, h, "noise" if i % 2 else "textured", 30, seed=300 + i) for i in range(n)]
    outs = [orc.oracle_encode(*R.to_planar(p, R.RGB24, cf), chroma_format=cf, want_coefs=True) for p in pics]
    with encoder(cf, n) as e:
        base = pipeline_launches(e)
        for fmt in R.FORMATS:
            fr = Frames()
            descs = [R.place_rgb(fr, R.as_format(p, fmt, seed=i), fmt, odd_pitch(R.BYTES_PER_PIXEL[fmt] * w, i), shift=i) for i, p in enumerate(pics)]
            torch.cuda.synchronize()
            before = e.kernel_launches
            e.submit_device_rgb(0, fmt, descs)
            for i, (_, dbg, coefs) in enumerate(outs):
                info = e.frame_info(0, i)
                assert (info.mcu_w, info.mcu_h, info.qscale, info.mb_var_sum) == (dbg.mcu_w, dbg.mcu_h, dbg.qscale, dbg.mb_var_sum)
                assert (info.header_bytes, info.scan_bits) == (dbg.header_bytes, dbg.scan_bits)
                assert (e.coefficients(0, i, coefs.shape[0]) == coefs).all()
            assert e.collect(0).jpegs == [o[0] for o in outs], R.NAMES[fmt]
            assert e.kernel_launches - before == base + 1, R.NAMES[fmt]


@pytest.mark.parametrize("kw", [{"range_mode": 1}, {"fixed_qscale": 3}])
@pytest.mark.parametrize("cf", [0, 1, 2])
def test_range_mode_does_not_apply_and_fixed_qscale_does(orc, cf, kw):
    import torch

    fr = Frames()
    geoms = [(322, 242), (1918, 1078), (131, 77)]
    pics = [picture(orc, w, h, "textured", 70, seed=500 + i) for i, (w, h) in enumerate(geoms)]
    want = [want_jpeg(orc, p, cf, fixed_qscale=kw.get("fixed_qscale", 0), range_mode=0) for p in pics]
    with encoder(cf, len(geoms), **kw) as e:
        for fmt in (R.RGB24, R.BGRX, R.PLANAR):
            descs = [R.place_rgb(fr, R.as_format(p, fmt), fmt, shift=i) for i, p in enumerate(pics)]
            torch.cuda.synchronize()
            e.submit_device_rgb(0, fmt, descs)
            assert e.collect(0).jpegs == want, (R.NAMES[fmt], kw)
            assert e.rgb2jpeg(R.as_format(pics[0], fmt), fmt) == want[0]


def test_64_1080p_rgb24_frames(orc):
    """64 x 1080p RGB24 in one allocation, one submit: first, last and six random frames against the oracle"""
    import h2j_b200 as h2j

    n, w, h = 64, 1920, 1080
    bases = [picture(orc, w, h, "textured" if i % 2 else "noise", 20 + 5 * i, seed=900 + i) for i in range(8)]
    rng = random.Random(64)
    pick = [rng.randrange(8) for _ in range(n)]
    stride = align(3 * w * h, 256)
    d, ptr = upload([bases[i].reshape(-1) for i in pick], stride)
    descs = [h2j.FrameDesc(ptr + i * stride, w, h, 3 * w, 0, 0, 0) for i in range(n)]
    check = sorted({0, n - 1} | set(rng.sample(range(1, n - 1), 6)))
    with h2j.Encoder(max_width=w, max_height=h, max_batch=n, n_slots=1) as e:
        e.submit_device_rgb(0, h2j.RGB_RGB24, descs)
        got = e.collect(0).jpegs
    for i in check:
        assert got[i] == want_jpeg(orc, bases[pick[i]], 0), i


@pytest.fixture(scope="module")
def every_triple():
    """a 4096 x 4096 picture that holds every RGB triple exactly once, in a shuffled order"""
    idx = np.random.default_rng(24).permutation(1 << 24)
    return np.stack([idx >> 16, (idx >> 8) & 255, idx & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)


@pytest.mark.parametrize("cf", [0, 2])
def test_every_triple_converts_exactly(every_triple, cf):
    """the planes the pipeline read equal C(frame) bit for bit: at 4:4:4 the conversion alone, at 4:2:0 with the boxes"""
    import torch

    want = R.to_planar(every_triple, R.RGB24, cf)
    with encoder(cf, 1, max_width=4096, max_height=4096, fixed_qscale=31, max_jpeg_bytes=64 << 20) as e:
        for fmt in R.FORMATS:
            fr = Frames()
            d = R.place_rgb(fr, R.as_format(every_triple, fmt, seed=fmt), fmt, shift=fmt)
            torch.cuda.synchronize()
            e.submit_device_rgb(0, fmt, [d])
            e.wait(0)
            got = e.frame_planes(0, 0, 4096, 4096)
            for k in range(3):
                assert (got[k] == want[k]).all(), (R.NAMES[fmt], "YUV"[k], int((got[k] != want[k]).sum()))
            assert e.collect(0).status == [0]


def test_frame_planes_of_other_inputs(orc):
    """the hook answers for a downscaled frame (D_k), a P010 frame (the truncation), and I420 and NV12 frames read in place"""
    import torch

    import h2j_b200 as h2j

    w, h = 640, 362  # rows on 8-byte boundaries: the I420 and NV12 frames are read in place
    y, u, v = orc.synth_planes_fmt(w, h, 0, "noise", seed=31, amp=90)
    fr = Frames()
    i420 = desc(fr, y, u, v, *planar(y, u))
    nv12 = desc(fr, y, u, v, *semiplanar(y, 704))
    words = [p.astype(np.uint16) << 8 | np.uint16(0xC0) for p in (y, u, v)]  # 10-bit values p * 4 + 3, MSB-aligned (P010)
    p010 = place(*words, *semiplanar(words[0], 2 * 704))
    d16, p16 = upload([p010], align(p010.size, 256))
    torch.cuda.synchronize()

    def planes_equal(got, want, what):
        for k in range(3):
            assert (got[k] == want[k]).all(), (what, "YUV"[k])

    with encoder(0, 1) as e:
        e.submit_device_downscaled(0, h2j.LAYOUT_PLANAR, [i420], 4)
        e.wait(0)
        planes_equal(e.frame_planes(0, 0, *h2j.downscaled_size(w, h, 4)), downscale_planar(y, u, v, 4), "1/4")
        e.collect(0)
        e.submit_device_semiplanar16(0, p16, align(p010.size, 256), 2 * 704, 2 * 704 * h, 16, 1, w, h)
        e.wait(0)
        planes_equal(e.frame_planes(0, 0, w, h), (y, u, v), "P010")
        e.collect(0)
        for layout, d in ((h2j.LAYOUT_PLANAR, i420), (h2j.LAYOUT_SEMIPLANAR, nv12)):
            e.submit_device_list(0, layout, [d])
            e.collect(0)
            planes_equal(e.frame_planes(0, 0, w, h), (y, u, v), layout)
        with pytest.raises(h2j.H2JError) as ex:
            e.frame_planes(0, 0, w + 16, h)
        assert ex.value.status == h2j.ERR_INVALID_ARG
        L = e._lib
        assert L.h2j_debug_frame_planes(e._h, 0, 1, None, None, None) == h2j.ERR_INVALID_ARG


def test_host_pictures(orc):
    """h2j_encode_frame_rgb on a packed view with a row stride wider than its row, a planar CHW array and three planes of
    their own, from pageable and pinned memory; its staging is shared with h2j_encode_frame16 and grows as needed"""
    import torch

    import h2j_b200 as h2j

    w, h = 1280, 720
    rgb = picture(orc, w, h, "textured", 50, seed=41)
    want = want_jpeg(orc, rgb, 0)
    y, u, v = orc.synth_planes(w, h, "textured", seed=42)
    want16 = orc.oracle_encode(y, u, v)[0]
    words = [p.astype(np.uint16) << 2 for p in (y, u, v)]
    wide = np.zeros((h, w + 37, 4), np.uint8)
    wide[:, :w] = R.as_format(rgb, R.BGRX, seed=3)
    pinned = h2j.PinnedBuffer(3 * w * h)
    pinned.array[:] = R.as_format(rgb, R.RGB24).reshape(-1)
    chw = R.as_format(rgb, R.PLANAR)
    fr = Frames()
    with encoder(0, 1) as e:
        assert e.yuv2jpeg16(*words, 10) == want16  # the staging at its 16-bit size ...
        assert e.rgb2jpeg(wide[:, :w], R.BGRX) == want  # ... grown for 4 bytes a pixel
        assert e.yuv2jpeg16(*words, 10) == want16
        assert e.rgb2jpeg(pinned.array.reshape(h, w, 3), R.RGB24) == want
        assert e.rgb2jpeg(chw, R.PLANAR) == want
        assert e.rgb2jpeg([np.ascontiguousarray(chw[k]) for k in range(3)], R.PLANAR) == want
        assert e.rgb2jpeg(np.ascontiguousarray(rgb[..., ::-1]), R.BGR24) == want
        planes = e.frame_planes(0, 0, w, h)
        for k, p in enumerate(R.to_planar(rgb, R.RGB24, 0)):
            assert (planes[k] == p).all()
        d = R.place_rgb(fr, R.as_format(rgb, R.RGBX), R.RGBX)
        torch.cuda.synchronize()
        e.submit_device_rgb(0, R.RGBX, [d])
        assert e.collect(0).jpegs == [want]
    pinned.free()


def test_rgb_and_yuv_batches_in_flight_together(orc):
    import torch

    import h2j_b200 as h2j

    fr = Frames()
    n = 4
    pics = [picture(orc, 1920, 1080, "textured" if i % 2 else "noise", 30, seed=800 + i) for i in range(n)]
    yuvs = [orc.synth_planes(1920, 1080, "textured", seed=810 + i) for i in range(n)]
    rgb_descs = [R.place_rgb(fr, R.as_format(p, R.BGRX, seed=i), R.BGRX, 7680) for i, p in enumerate(pics)]
    yuv_descs = [desc(fr, y, u, v, *semiplanar(y, 2048, 8)) for y, u, v in yuvs]
    torch.cuda.synchronize()
    with h2j.Encoder(max_width=1920, max_height=1088, max_batch=n, n_slots=2) as e:
        e.submit_device_rgb(0, h2j.RGB_BGRX, rgb_descs)
        e.submit_device_list(1, h2j.LAYOUT_SEMIPLANAR, yuv_descs)
        yuv = e.collect(1).jpegs
        rgb = e.collect(0).jpegs
    assert rgb == [want_jpeg(orc, p, 0) for p in pics]
    assert yuv == [orc.oracle_encode(*p)[0] for p in yuvs]


# ---- argument checks ------------------------------------------------------------------------------------------------
W, H, B = 64, 32, 2  # the encoder's maximum and batch


def malformed_cases():
    """(entry point, what is wrong, overrides, expected status); every frame is valid unless the overrides say otherwise"""
    import h2j_b200

    INV, UNS = h2j_b200.ERR_INVALID_ARG, h2j_b200.ERR_UNSUPPORTED
    cases = []
    for fmt in R.FORMATS:
        row = R.BYTES_PER_PIXEL[fmt] * W
        cases += [
            ("device", "slot -1", dict(fmt=fmt, slot=-1), INV),
            ("device", "slot past n_slots", dict(fmt=fmt, slot=2), INV),
            ("device", "null frames", dict(fmt=fmt, frames=None), INV),
            ("device", "n 0", dict(fmt=fmt, n=0), INV),
            ("device", "n past max_batch", dict(fmt=fmt, n=B + 1), INV),
            ("device", "null frame data", dict(fmt=fmt, data=0), INV),
            ("device", "null data in the second frame only", dict(fmt=fmt, null_frame=True), INV),
            ("device", "pitch shorter than a row", dict(fmt=fmt, pitch=row - 1), INV),
            ("device", "1 pixel wide", dict(fmt=fmt, w=1), UNS),
            ("device", "1 pixel high", dict(fmt=fmt, hh=1), UNS),
            ("device", "wider than the maximum", dict(fmt=fmt, w=2 * W, pitch=2 * row), UNS),
            ("device", "taller than the maximum", dict(fmt=fmt, hh=2 * H), UNS),
            ("device", "wider than 65500 pixels", dict(fmt=fmt, w=70000, pitch=70000 * R.BYTES_PER_PIXEL[fmt]), UNS),
            ("host", "null planes", dict(fmt=fmt, planes=None), INV),
            ("host", "null out", dict(fmt=fmt, out_ok=False), INV),
            ("host", "stride shorter than a row", dict(fmt=fmt, strides=(row - 1, row, row)), INV),
            ("host", "1 pixel wide", dict(fmt=fmt, w=1), UNS),
            ("host", "wider than the maximum", dict(fmt=fmt, w=2 * W, strides=(2 * row,) * 3), UNS),
            ("host", "taller than the maximum", dict(fmt=fmt, hh=2 * H), UNS),
        ]
    for bad in (-1, 5, 99):
        cases += [("device", f"format {bad}", dict(fmt=bad), INV), ("host", f"format {bad}", dict(fmt=bad), INV)]
    cases += [
        ("device", "G plane inside the R plane", dict(fmt=R.PLANAR, u_off=W * H - 1), INV),
        ("device", "B plane inside the R plane", dict(fmt=R.PLANAR, v_off=W * H - 1), INV),
        ("device", "B plane at the R plane's start", dict(fmt=R.PLANAR, v_off=0), INV),
        ("host", "null G plane", dict(fmt=R.PLANAR, null_plane=1), INV),
        ("host", "null B plane", dict(fmt=R.PLANAR, null_plane=2), INV),
        ("host", "short G stride", dict(fmt=R.PLANAR, strides=(W, W - 1, W)), INV),
        ("host", "short B stride", dict(fmt=R.PLANAR, strides=(W, W, W - 1)), INV),
    ]
    return cases


def test_malformed_rgb_calls_leave_the_slot_as_it_was():
    """every malformed call returns its status; a batch in flight on the other slot stays collectable with its JPEGs, the
    last batch keeps its frame_info, and nothing is left in flight"""
    import torch

    import h2j_b200

    rng = np.random.default_rng(12)
    host_buf = rng.integers(0, 256, 1 << 16, dtype=np.uint8)
    dev = torch.from_numpy(rng.integers(0, 256, 1 << 16, dtype=np.uint8)).cuda()
    torch.cuda.synchronize()
    S = 4 * W * H * 3  # bytes between the frames of a call: any format at twice the maximum width
    out = np.empty(1 << 20, np.uint8)
    size = C.c_size_t(0)

    with h2j_b200.Encoder(max_width=W, max_height=H, max_batch=B, n_slots=2) as e:
        L, hd = e._lib, e._h

        def device(fmt, slot=0, frames="ok", n=B, data=None, null_frame=False, pitch=None, w=W, hh=H, u_off=None, v_off=None):
            p = dev.data_ptr() if data is None else data
            pitch = pitch or R.BYTES_PER_PIXEL.get(fmt, 3) * w
            u_off = pitch * hh if u_off is None else u_off
            v_off = 2 * pitch * hh if v_off is None else v_off
            ptrs = [p + i * S if p else 0 for i in range(B)]
            if null_frame:
                ptrs[1] = 0
            d = (h2j_b200.FrameDesc * B)(*[h2j_b200.FrameDesc(q, w, hh, pitch, 0, u_off, v_off) for q in ptrs])
            rc = L.h2j_submit_device_rgb(hd, slot, fmt, None if frames is None else d, n)
            if rc == 0:
                e._n_in_slot[slot] = n  # what collect() sizes its buffers by
            return rc

        def host(fmt, planes="ok", out_ok=True, strides=None, w=W, hh=H, null_plane=None):
            row = R.BYTES_PER_PIXEL.get(fmt, 3) * w
            ptrs = (C.c_void_p * 3)(*[None if k == null_plane else host_buf.ctypes.data + k * row * hh for k in range(3)])
            st = (C.c_int * 3)(*(strides or (row, row, row)))
            return L.h2j_encode_frame_rgb(hd, fmt, None if planes is None else ptrs, st, w, hh, out.ctypes.data if out_ok else None, out.size,
                                          C.byref(size))

        def info_bytes(i):
            info = e.frame_info(0, i)
            return C.string_at(C.addressof(info), C.sizeof(info))

        assert device(R.RGB24, w=48, hh=16) == 0
        want = e.collect(0)
        assert want.status == [0, 0]
        infos = [info_bytes(i) for i in range(2)]

        # a batch in flight: a valid call of either entry point on its slot is refused, and the batch stays collectable
        assert device(R.RGB24, w=48, hh=16) == 0
        for fmt in R.FORMATS:
            assert device(fmt) == h2j_b200.ERR_BUSY and host(fmt) == h2j_b200.ERR_BUSY, R.NAMES[fmt]
        got = e.collect(0)
        assert got.jpegs == want.jpegs and [info_bytes(i) for i in range(2)] == infos

        # every malformed call on slot 0 returns its status, with a batch in flight on slot 1
        assert device(R.RGB24, slot=1, w=48, hh=16) == 0
        wrong = []
        for name, what, kw, status in malformed_cases():
            rc = (device if name == "device" else host)(**kw)
            if rc != status:
                wrong.append(f"{name}, {R.NAMES.get(kw['fmt'], kw['fmt'])}, {what}: status {rc}, expected {status}")
        assert not wrong, "\n".join(wrong)
        got = e.collect(1)
        assert got.jpegs == want.jpegs and got.status == want.status
        assert [info_bytes(i) for i in range(2)] == infos, "a rejected call changed the last batch's frame_info"
        with pytest.raises(h2j_b200.H2JError) as ei:
            e.collect(0)  # nothing in flight: no rejected call left the slot busy
        assert ei.value.status == h2j_b200.ERR_BUSY

        # and the valid calls the table starts from are accepted
        for fmt in R.FORMATS:
            assert device(fmt) == 0, R.NAMES[fmt]
            assert e.collect(0).status == [0] * B
            assert host(fmt) == 0, R.NAMES[fmt]


# ---- decode-back sanity with an independent decoder -------------------------------------------------------------------
def _decode(jpeg):
    import io

    Image = pytest.importorskip("PIL.Image")
    return np.asarray(Image.open(io.BytesIO(jpeg)).convert("RGB")).astype(np.int64)


@pytest.mark.parametrize("colour", [(255, 0, 0), (0, 255, 0), (0, 0, 255), (255, 255, 255), (40, 90, 200)])
@pytest.mark.parametrize("fmt", [R.RGB24, R.BGR24, R.BGRX, R.PLANAR])
def test_flat_colours_decode_to_themselves(colour, fmt):
    """channel order and Cb / Cr order: a flat frame decodes to its colour (within the matrices' rounding)"""
    rgb = np.empty((64, 96, 3), np.uint8)
    rgb[:] = colour
    with encoder(0, 1, fixed_qscale=1) as e:
        got = _decode(e.rgb2jpeg(R.as_format(rgb, fmt), fmt))
    assert np.abs(got - np.array(colour)).max() <= 2, (colour, got[0, 0])


@pytest.mark.parametrize("cf", [0, 1, 2])
def test_smooth_content_decodes_close(orc, cf):
    """smooth content at fixed_qscale 1 decodes to a PSNR above 44 dB"""
    yy, xx = np.mgrid[0:240, 0:320].astype(np.float64)
    rgb = np.stack([128 + 100 * np.sin(xx / 40), 128 + 100 * np.cos(yy / 30), 128 + 80 * np.sin((xx + yy) / 50)], -1).astype(np.uint8)
    with encoder(cf, 1, fixed_qscale=1) as e:
        got = _decode(e.rgb2jpeg(rgb, R.RGB24))
    mse = ((got - rgb.astype(np.int64)) ** 2).mean()
    assert 10 * np.log10(255 ** 2 / mse) > 44, mse
