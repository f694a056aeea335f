"""GPU suite: resized device frames (h2j_submit_device_resized).  The frames the input stage writes must equal the numpy
model of R(frame) (tests/support/resize.py, pinned against Pillow on the CPU) bit for bit, and every JPEG must be
byte-identical to the oracle's JPEG of those planes, with the same encoder settings.  Sources sit in their own allocations
surrounded by 0xA5 padding, and pitch and surface gaps are 0xA5 too: a padding byte that reached a sum would change a sample."""
import ctypes as C
import random

import numpy as np
import pytest

from tests.support.layouts import Frames, align, desc, encoder, place, planar, semiplanar, upload
from tests.support.resize import FILTERS, resize_planar

pytestmark = pytest.mark.gpu

# (source w, h, kind, amp) -> output (W, H): odd sizes, upscales, one axis changed, the identity, 2/3, 1/3, 1/6, 224x224
RESIZES = [((16, 16, "textured", 40), (16, 16)), ((2, 2, "noise", 100), (7, 5)), ((17, 17, "noise", 60), (9, 33)),
           ((33, 47, "blocks", 30), (33, 20)), ((131, 77, "textured", 80), (262, 77)), ((64, 64, "binary", 0), (31, 97)),
           ((322, 242, "textured", 40), (215, 161)), ((641, 479, "noise", 20), (224, 224)), ((9, 31, "noise", 50), (2, 2)),
           ((1280, 720, "textured", 30), (427, 240)), ((1920, 1080, "textured", 40), (320, 180)),
           ((1918, 1078, "textured", 40), (1280, 720)), ((854, 480, "ff", 0), (1280, 720))]

_planes = {}


def source(orc, w, h, fmt, kind="textured", amp=40, seed=0):
    key = (w, h, fmt, kind, amp, seed)
    if key not in _planes:
        _planes[key] = orc.synth_planes_fmt(w, h, fmt, kind, seed=seed, amp=amp)
    return _planes[key]


def odd_pitch(n, j):
    return n + 1 + (n % 2) + 2 * j


def layouts(h2j, fr, y, u, v, i):
    """(name, layout, desc) of one source frame at every layout the suite covers"""
    h, w = y.shape
    ch, cw = u.shape
    sp_row = max(w, 2 * cw)
    return [
        ("planar tight", h2j.LAYOUT_PLANAR, desc(fr, y, u, v, *planar(y, u))),
        ("planar decoder", h2j.LAYOUT_PLANAR, desc(fr, y, u, v, *planar(y, u, align(w, 256), align(cw, 256), align(h, 16) - h + 16))),
        ("planar shifted", h2j.LAYOUT_PLANAR, desc(fr, y, u, v, *planar(y, u, odd_pitch(w, i % 3), odd_pitch(cw, i % 2), i % 3), shift=1 + i % 15)),
        ("semi-planar aligned", h2j.LAYOUT_SEMIPLANAR, desc(fr, y, u, v, *semiplanar(y, align(sp_row, 64), align(h, 16) - h))),
        ("semi-planar unaligned", h2j.LAYOUT_SEMIPLANAR, desc(fr, y, u, v, *semiplanar(y, odd_pitch(sp_row, i % 2), 1), shift=1 + (i + 4) % 15)),
    ]


def check_planes(e, slot, i, W, H, want):
    got = e.frame_planes(slot, i, W, H)
    for name, g, wnt in zip("yuv", got, want):
        assert g.shape == wnt.shape and np.array_equal(g, wnt), (i, W, H, name, int(np.abs(g.astype(int) - wnt).max()))


@pytest.mark.parametrize("flt", FILTERS)
@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_every_layout_as_a_mixed_list(orc, fmt, flt):
    """one list per layout that mixes all sizes (the list form of the pipeline): planes against the model, JPEGs against
    the oracle"""
    import torch

    import h2j_b200 as h2j

    fr = Frames()
    sizes, models, want, per_layout = [], [], [], {}
    for i, ((w, h, kind, amp), out) in enumerate(RESIZES):
        y, u, v = source(orc, w, h, fmt, kind, amp, seed=1200 + i)
        r = resize_planar(y, u, v, *out, fmt, flt)
        sizes.append(out)
        models.append(r)
        want.append(orc.oracle_encode(*r, chroma_format=fmt)[0])
        for name, layout, d in layouts(h2j, fr, y, u, v, i):
            per_layout.setdefault((name, layout), []).append(d)
    torch.cuda.synchronize()
    with encoder(fmt, len(RESIZES)) as e:
        for (name, layout), descs in per_layout.items():
            e.submit_device_resized(0, layout, descs, sizes, flt)
            e.wait(0)
            for i, (W, H) in enumerate(sizes):
                check_planes(e, 0, i, W, H, models[i])
            got = e.collect(0).jpegs
            for (W, H), g, wnt in zip(sizes, got, want):
                assert g == wnt, f"{W}x{H} fmt {fmt} filter {flt} {name}"


@pytest.mark.parametrize("layout", [0, 1])
def test_identity_equals_the_list_submit(orc, layout):
    import torch

    import h2j_b200 as h2j

    fr = Frames()
    srcs = [source(orc, w, h, 0, seed=1300 + i) for i, (w, h) in enumerate([(322, 242), (1283, 723), (64, 48)])]
    if layout == h2j.LAYOUT_PLANAR:
        descs = [desc(fr, y, u, v, *planar(y, u, odd_pitch(y.shape[1], i)), shift=i) for i, (y, u, v) in enumerate(srcs)]
    else:
        descs = [desc(fr, y, u, v, *semiplanar(y, align(max(y.shape[1], 2 * u.shape[1]), 64), 3)) for y, u, v in srcs]
    sizes = [(y.shape[1], y.shape[0]) for y, _, _ in srcs]
    torch.cuda.synchronize()
    with encoder(0, 3) as e:
        e.submit_device_list(0, layout, descs)
        listed = e.collect(0).jpegs
        for flt in FILTERS:
            e.submit_device_resized(0, layout, descs, sizes, flt)
            assert e.collect(0).jpegs == listed == [orc.oracle_encode(*p)[0] for p in srcs]


@pytest.mark.parametrize("kw", [{"range_mode": 1}, {"fixed_qscale": 3}])
@pytest.mark.parametrize("fmt", [0, 2])
def test_range_conversion_and_fixed_qscale(orc, fmt, kw):
    import torch

    import h2j_b200 as h2j

    fr = Frames()
    geoms = [((322, 242), (224, 224)), ((1918, 1078), (640, 360)), ((131, 77), (200, 150))]
    srcs = [source(orc, w, h, fmt, "textured", 70, seed=1400 + i) for i, ((w, h), _) in enumerate(geoms)]
    descs = [desc(fr, y, u, v, *semiplanar(y, odd_pitch(max(y.shape[1], 2 * u.shape[1]), i)), shift=i) for i, (y, u, v) in enumerate(srcs)]
    sizes = [o for _, o in geoms]
    torch.cuda.synchronize()
    with encoder(fmt, len(geoms), **kw) as e:
        for flt in (0, 2):
            e.submit_device_resized(0, h2j.LAYOUT_SEMIPLANAR, descs, sizes, flt)
            want = [orc.oracle_encode(*resize_planar(*p, *o, fmt, flt), chroma_format=fmt, **kw)[0] for p, o in zip(srcs, sizes)]
            assert e.collect(0).jpegs == want, (fmt, kw, flt)


@pytest.mark.parametrize("out", [(224, 224), (1280, 720)])
def test_64_decoder_layout_nv12_frames_in_one_submit(orc, out):
    """64 x 1080p NV12 at a hardware decoder's layout (pitch 2048, pair plane behind 1088 rows): the batch form"""
    import h2j_b200 as h2j

    n, pitch, surf = 64, 2048, 1088
    frame_bytes = pitch * surf * 3 // 2
    bases = [source(orc, 1920, 1080, 0, "textured" if i % 2 else "noise", 20 + 5 * i, seed=1500 + i) for i in range(8)]
    rng = random.Random(out[0])
    pick = [rng.randrange(8) for _ in range(n)]
    placed = [place(y, u, v, *semiplanar(y, pitch, surf - 1080), size=frame_bytes) for y, u, v in bases]
    d, ptr = upload([placed[i] for i in pick], frame_bytes)
    descs = [h2j.FrameDesc(ptr + i * frame_bytes, 1920, 1080, pitch, pitch, pitch * surf, 0) for i in range(n)]
    check = sorted({0, n - 1} | set(rng.sample(range(1, n - 1), 4)))
    with h2j.Encoder(max_width=1280, max_height=720, max_batch=n, n_slots=1) as e:
        e.submit_device_resized(0, h2j.LAYOUT_SEMIPLANAR, descs, [out] * n, h2j.FILTER_BICUBIC)
        got = e.collect(0).jpegs
    for i in check:
        assert got[i] == orc.oracle_encode(*resize_planar(*bases[pick[i]], *out, 0, 2))[0], i


def test_long_windows_and_spans_wider_than_the_staging_buffer(orc):
    """3840x2160 to 2x2 (every source sample in one window), 17x4098 to 5x3 (windows 1366 rows tall), 20000x4 to 3x2 (a
    luma row of 20000 samples and a row of 10000 pairs, staged in pieces)"""
    import torch

    import h2j_b200 as h2j

    fr = Frames()
    cases = [((3840, 2160), (2, 2)), ((17, 4098), (5, 3)), ((20000, 4), (3, 2)), ((20000, 4), (2400, 4))]
    srcs = [source(orc, w, h, 0, "textured", 60, seed=1600 + i) for i, ((w, h), _) in enumerate(cases)]
    sizes = [o for _, o in cases]
    with encoder(0, len(cases), max_width=2400, max_height=1088) as e:
        for layout in (h2j.LAYOUT_PLANAR, h2j.LAYOUT_SEMIPLANAR):
            if layout == h2j.LAYOUT_PLANAR:
                descs = [desc(fr, y, u, v, *planar(y, u, odd_pitch(y.shape[1], 0)), shift=3) for y, u, v in srcs]
            else:
                descs = [desc(fr, y, u, v, *semiplanar(y, odd_pitch(max(y.shape[1], 2 * u.shape[1]), 1), 2), shift=5) for y, u, v in srcs]
            torch.cuda.synchronize()
            for flt in FILTERS:
                models = [resize_planar(*p, *o, 0, flt) for p, o in zip(srcs, sizes)]
                e.submit_device_resized(0, layout, descs, sizes, flt)
                e.wait(0)
                for i, (W, H) in enumerate(sizes):
                    check_planes(e, 0, i, W, H, models[i])
                assert e.collect(0).jpegs == [orc.oracle_encode(*m)[0] for m in models], (layout, flt)


@pytest.mark.parametrize("layout", [0, 1])
def test_one_launch_more_than_the_pipeline(orc, layout):
    """a resized submit costs exactly one launch more than an in-place list submit of frames of the output size"""
    import torch

    import h2j_b200 as h2j

    fr = Frames()
    sizes = [(1280, 720), (1279, 719), (640, 360)]
    srcs = [source(orc, w, h, 0, seed=1700 + i) for i, (w, h) in enumerate(sizes)]
    y, u, v = resize_planar(*srcs[0], 224, 224, 0, 1)
    small = [desc(fr, y, u, v, *planar(y, u))] * 3
    if layout == h2j.LAYOUT_PLANAR:
        descs = [desc(fr, y, u, v, *planar(y, u), shift=3) for y, u, v in srcs]
    else:
        descs = [desc(fr, y, u, v, *semiplanar(y, 1283), shift=5) for y, u, v in srcs]
    torch.cuda.synchronize()
    with encoder(0, 3) as e:
        l0 = e.kernel_launches
        e.submit_device_list(0, h2j.LAYOUT_PLANAR, small)
        l_list = e.kernel_launches - l0
        e.collect(0)
        for batch, out in ((descs, [(224, 224), (225, 223), (100, 60)]), (descs, [(224, 224)] * 3)):  # list form, batch form
            l0 = e.kernel_launches
            e.submit_device_resized(0, layout, batch, out, h2j.FILTER_BILINEAR)
            assert e.kernel_launches - l0 == l_list + 1
            e.collect(0)
    assert l_list == 7


def test_thumbnail_encoder_argument_checks_leave_the_last_batch(orc):
    """an encoder sized for thumbnails takes 1080p sources; every refused call leaves the previous batch's JPEG, frame info
    and planes as they were"""
    import torch

    import h2j_b200 as h2j

    fr = Frames()
    y, u, v = source(orc, 1920, 1080, 0, seed=1800)
    src = desc(fr, y, u, v, *semiplanar(y, 2048, 8))
    ty, tu, tv = source(orc, 2, 2, 0, seed=1801)
    tiny = desc(fr, ty, tu, tv, *planar(ty, tu))
    torch.cuda.synchronize()
    with encoder(0, 2, max_width=480, max_height=272) as e:
        want = resize_planar(y, u, v, 480, 270, 0, 2)
        e.submit_device_resized(0, h2j.LAYOUT_SEMIPLANAR, [src], [(480, 270)], h2j.FILTER_BICUBIC)
        info0 = e.frame_info(0, 0)
        d_out, cap, sizes, status = e.collect_device(0)
        jpeg0 = orc.oracle_encode(*want)[0]
        assert list(status) == [0] and e.read_device(d_out, int(sizes[0])) == jpeg0
        lib, h = e._lib, e._h

        def call(layout, descs, ws, hs, flt, n=None):
            n = len(descs) if n is None else n
            arr = (h2j.FrameDesc * max(1, len(descs)))(*descs)
            cw = None if ws is None else (C.c_int * max(1, len(ws)))(*ws)
            ch = None if hs is None else (C.c_int * max(1, len(hs)))(*hs)
            return lib.h2j_submit_device_resized(h, 0, layout, arr, n, cw, ch, flt)

        sp, pl = h2j.LAYOUT_SEMIPLANAR, h2j.LAYOUT_PLANAR
        bad = h2j.FrameDesc(src.data, 1920, 1080, 1000, 2048, 2048 * 1088, 0)
        null = h2j.FrameDesc(None, 1920, 1080, 2048, 2048, 2048 * 1088, 0)
        big = h2j.FrameDesc(src.data, 65501, 2, 65504, 65504, 65504 * 2, 0)
        table = [
            ("null out_widths", (sp, [src], None, [100], 0), h2j.ERR_INVALID_ARG),
            ("null out_heights", (sp, [src], [100], None, 0), h2j.ERR_INVALID_ARG),
            ("filter -1", (sp, [src], [100], [100], -1), h2j.ERR_INVALID_ARG),
            ("filter 3", (sp, [src], [100], [100], 3), h2j.ERR_INVALID_ARG),
            ("n 0", (sp, [src], [100], [100], 0, 0), h2j.ERR_INVALID_ARG),
            ("n past max_batch", (sp, [src] * 3, [100] * 3, [100] * 3, 0), h2j.ERR_INVALID_ARG),
            ("bad layout", (2, [src], [100], [100], 0), h2j.ERR_INVALID_ARG),
            ("null data in the second frame", (sp, [src, null], [100, 100], [100, 100], 0), h2j.ERR_INVALID_ARG),
            ("pitch shorter than a luma row", (sp, [bad], [100], [100], 0), h2j.ERR_INVALID_ARG),
            ("planar frame as pairs: short pair rows", (sp, [src, tiny], [100, 100], [100, 100], 0), h2j.ERR_INVALID_ARG),
            ("output 1 wide", (sp, [src], [1], [100], 0), h2j.ERR_UNSUPPORTED),
            ("output 1 high", (sp, [src], [100], [1], 0), h2j.ERR_UNSUPPORTED),
            ("output 65501 wide", (sp, [src], [65501], [100], 0), h2j.ERR_UNSUPPORTED),
            ("output wider than the maximum", (sp, [src], [481], [100], 0), h2j.ERR_UNSUPPORTED),
            ("output taller than the maximum, second frame", (sp, [src, src], [100, 100], [100, 273], 0), h2j.ERR_UNSUPPORTED),
            ("source wider than 65500", (pl, [big], [100], [2], 0), h2j.ERR_UNSUPPORTED),
        ]
        for name, args, code in table:
            assert call(*args) == code, name
            info = e.frame_info(0, 0)
            assert (info.qscale, info.scan_bits, info.mcu_w, info.mcu_h) == (info0.qscale, info0.scan_bits, info0.mcu_w, info0.mcu_h), name
            assert e.read_device(d_out, int(sizes[0])) == jpeg0, name
            check_planes(e, 0, 0, 480, 270, want)
        # a 2x2 source upscaled to the maximum, and the busy slot
        e.submit_device_resized(0, pl, [tiny], [(480, 272)], h2j.FILTER_BILINEAR)
        with pytest.raises(h2j.H2JError) as ex:
            e.submit_device_resized(0, pl, [tiny], [(480, 272)], h2j.FILTER_BILINEAR)
        assert ex.value.status == h2j.ERR_BUSY
        assert e.collect(0).jpegs == [orc.oracle_encode(*resize_planar(ty, tu, tv, 480, 272, 0, 1))[0]]


def test_resized_and_downscaled_batches_in_flight_on_two_slots(orc):
    import torch

    import h2j_b200 as h2j
    from tests.support.downscale import downscale_planar

    fr = Frames()
    n = 4
    srcs = [source(orc, 1920, 1080, 0, "textured" if i % 2 else "noise", 30, seed=1900 + i) for i in range(n)]
    descs = [desc(fr, y, u, v, *semiplanar(y, 2048, 8)) for y, u, v in srcs]
    torch.cuda.synchronize()
    with h2j.Encoder(max_width=1920, max_height=1088, max_batch=n, n_slots=2, max_jpeg_bytes=8 * 1024 * 1024) as e:
        e.submit_device_resized(0, h2j.LAYOUT_SEMIPLANAR, descs, [(640, 360)] * n, h2j.FILTER_BILINEAR)
        e.submit_device_downscaled(1, h2j.LAYOUT_SEMIPLANAR, descs, 4)
        thumbs = e.collect(1).jpegs
        resized = e.collect(0).jpegs
    assert resized == [orc.oracle_encode(*resize_planar(*p, 640, 360, 0, 1))[0] for p in srcs]
    assert thumbs == [orc.oracle_encode(*downscale_planar(*p, 4))[0] for p in srcs]


def table_bytes(w_in, w_out):
    """bytes of BICUBIC coefficients of the axes w_in (array) -> w_out, as the library counts Pillow's windows"""
    w_in = np.asarray(w_in, np.float64)
    scale = w_in / w_out
    support = 2.0 * np.maximum(scale, 1.0)
    taps = 0
    for o in range(w_out):
        center = (o + 0.5) * scale
        taps = taps + np.minimum(np.trunc(center + support + 0.5), w_in) - np.maximum(np.trunc(center - support + 0.5), 0)
    return 4 * taps


def test_tables_larger_than_the_device_are_refused_and_the_encoder_stays_usable(orc):
    """131070 frames whose (source, output) pairs differ on every axis need about twice the device's memory for their
    coefficient tables: the submit returns ERR_NOMEM before it enqueues anything (the device buffer is asked for first, so
    no host memory is pinned), and the next submit works"""
    import torch

    import h2j_b200 as h2j

    n, side, per = 131070, 65500, 30
    y_bytes, c_side = side * side, (side + 1) // 2
    i = np.arange(n)
    a, b = np.divmod(i, per)
    w = side - 2 * a
    need = sum(int((table_bytes(w[b == k], 5 + 2 * k) * 2 + table_bytes((w[b == k] + 1) // 2, 3 + k) * 2).sum()) for k in range(per))
    assert need > 1.5 * torch.cuda.get_device_properties(0).total_memory, need
    buf = torch.empty(y_bytes + 2 * c_side * c_side, dtype=torch.uint8, device="cuda")
    descs = [h2j.FrameDesc(buf.data_ptr(), int(w[j]), int(w[j]), side, c_side, y_bytes, y_bytes + c_side * c_side) for j in range(n)]
    sizes = [(5 + 2 * int(b[j]), 5 + 2 * int(b[j])) for j in range(n)]
    fr = Frames()
    y, u, v = source(orc, 322, 242, 0, seed=2000)
    ok = desc(fr, y, u, v, *planar(y, u))
    torch.cuda.synchronize()
    with h2j.Encoder(max_width=64, max_height=64, max_batch=n, n_slots=1, max_jpeg_bytes=16384) as e:
        with pytest.raises(h2j.H2JError) as ex:
            e.submit_device_resized(0, h2j.LAYOUT_PLANAR, descs, sizes, h2j.FILTER_BICUBIC)
        assert ex.value.status == h2j.ERR_NOMEM
        del buf
        e.submit_device_resized(0, h2j.LAYOUT_PLANAR, [ok], [(63, 47)], h2j.FILTER_BICUBIC)
        assert e.collect(0).jpegs == [orc.oracle_encode(*resize_planar(y, u, v, 63, 47, 0, 2))[0]]
