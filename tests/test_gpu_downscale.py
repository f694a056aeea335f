"""GPU suite: downscaled device frames (h2j_submit_device_downscaled).  Every JPEG must be byte-identical to the oracle's
JPEG of the planar frame D_k(source) (tests/support/downscale.py), with the same encoder settings.  Sources sit in their own
allocations surrounded by 0xA5 padding, and pitch and surface gaps are 0xA5 too: a padding byte that reached an average
would change the JPEG."""
import random

import pytest

from tests.support.downscale import FACTORS, downscale_planar
from tests.support.layouts import CASES, Frames, align, desc, encoder, place, planar, semiplanar, upload

pytestmark = pytest.mark.gpu

GEOMETRIES = CASES + [(17, 4098, "textured", 40), (3840, 2160, "textured", 30)]
MAX_W, MAX_H = 1920, 2052  # the largest downscaled frames: 3840x2160 and 17x4098 at 1/2

_planes = {}


def source(orc, w, h, fmt, kind="textured", amp=40, seed=0):
    key = (w, h, fmt, kind, amp, seed)
    if key not in _planes:
        _planes[key] = orc.synth_planes_fmt(w, h, fmt, kind, seed=seed, amp=amp)
    return _planes[key]


def want_jpeg(orc, y, u, v, k, fmt, **kw):
    return orc.oracle_encode(*downscale_planar(y, u, v, k), chroma_format=fmt, **kw)[0]


def fits(w, h, k):
    return -(-w // k) >= 2 and -(-h // k) >= 2


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


@pytest.mark.parametrize("k", FACTORS)
@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_every_geometry_and_layout(orc, fmt, k):
    """one list per layout that mixes all sizes (the list form of the pipeline), every frame against the oracle"""
    import torch

    import h2j_b200 as h2j

    geoms = [g for g in GEOMETRIES if fits(g[0], g[1], k)]
    fr = Frames()
    want, per_layout = [], {}
    for i, (w, h, kind, amp) in enumerate(geoms):
        y, u, v = source(orc, w, h, fmt, kind, amp, seed=200 + i)
        want.append(want_jpeg(orc, y, u, v, k, fmt))
        for name, layout, d in layouts(h2j, fr, y, u, v, i):
            per_layout.setdefault((name, layout), []).append(d)
    torch.cuda.synchronize()
    with encoder(fmt, len(geoms), max_width=MAX_W, max_height=MAX_H) as e:
        for (name, layout), descs in per_layout.items():
            e.submit_device_downscaled(0, layout, descs, k)
            got = e.collect(0).jpegs
            for (w, h, _, _), g, wnt in zip(geoms, got, want):
                assert g == wnt, f"{w}x{h} fmt {fmt} 1/{k} {name}"


@pytest.mark.parametrize("k", FACTORS)
@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_uniform_list_runs_the_batch_form(orc, fmt, k):
    """frames of one downscaled size at their own addresses: the batch form, whose frame info matches the oracle's"""
    import torch

    import h2j_b200 as h2j

    w, h, n = 1283, 723, 4
    fr = Frames()
    srcs = [source(orc, w, h, fmt, "noise" if i % 2 else "textured", 30, seed=300 + i) for i in range(n)]
    outs = [orc.oracle_encode(*downscale_planar(*p, k), chroma_format=fmt, want_coefs=True) for p in srcs]
    flat = [desc(fr, y, u, v, *planar(y, u, odd_pitch(w, i)), shift=i) for i, (y, u, v) in enumerate(srcs)]
    semi = [desc(fr, y, u, v, *semiplanar(y, align(max(w, 2 * u.shape[1]), 256), 13)) for y, u, v in srcs]
    torch.cuda.synchronize()
    with encoder(fmt, n, max_width=MAX_W, max_height=MAX_H) as e:
        for layout, descs in ((h2j.LAYOUT_PLANAR, flat), (h2j.LAYOUT_SEMIPLANAR, semi)):
            e.submit_device_downscaled(0, layout, descs, k)
            for i, (_, dbg, coefs) in enumerate(outs):
                info = e.frame_info(0, i)
                assert (info.mcu_w, info.mcu_h, info.qscale, info.mb_var_sum) == (dbg.mcu_w, dbg.mcu_h, dbg.qscale, dbg.mb_var_sum)
                assert (info.header_bytes, info.scan_bits) == (dbg.header_bytes, dbg.scan_bits)
                assert (e.coefficients(0, i, coefs.shape[0]) == coefs).all()
            assert e.collect(0).jpegs == [o[0] for o in outs], (fmt, k, layout)


def test_debug_hooks_answer_for_the_downscaled_frame_of_a_mixed_list(orc):
    import torch

    import h2j_b200 as h2j

    sizes = [(1920, 1080), (66, 94), (641, 479)]
    fr = Frames()
    descs, outs = [], []
    for i, (w, h) in enumerate(sizes):
        y, u, v = source(orc, w, h, 0, seed=400 + i)
        outs.append(orc.oracle_encode(*downscale_planar(y, u, v, 2), want_coefs=True))
        descs.append(desc(fr, y, u, v, *planar(y, u), shift=i))
    torch.cuda.synchronize()
    with encoder(0, len(sizes)) as e:
        e.submit_device_downscaled(0, h2j.LAYOUT_PLANAR, descs, 2)
        for i, (_, dbg, coefs) in enumerate(outs):
            info = e.frame_info(0, i)
            assert (info.mcu_w, info.mcu_h, info.qscale, info.scan_bits) == (dbg.mcu_w, dbg.mcu_h, dbg.qscale, dbg.scan_bits)
            for t in range(4):
                assert list(info.hist[t]) == list(dbg.hist[t])
            assert (e.coefficients(0, i, coefs.shape[0]) == coefs).all()
        assert e.collect(0).jpegs == [o[0] for o in outs]


@pytest.mark.parametrize("kw", [{"range_mode": 1}, {"fixed_qscale": 3}])
@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_range_conversion_and_fixed_qscale(orc, fmt, kw):
    import torch

    import h2j_b200 as h2j

    fr = Frames()
    geoms = [(322, 242), (1918, 1078), (131, 77)]
    srcs = [source(orc, w, h, fmt, "textured", 70, seed=500 + i) for i, (w, h) in enumerate(geoms)]
    descs = [desc(fr, y, u, v, *semiplanar(y, odd_pitch(max(y.shape[1], 2 * u.shape[1]), i)), shift=i) for i, (y, u, v) in enumerate(srcs)]
    torch.cuda.synchronize()
    with encoder(fmt, len(geoms), **kw) as e:
        for k in (2, 4):
            e.submit_device_downscaled(0, h2j.LAYOUT_SEMIPLANAR, descs, k)
            assert e.collect(0).jpegs == [want_jpeg(orc, *p, k, fmt, **kw) for p in srcs], (fmt, kw, k)


@pytest.mark.parametrize("layout", [0, 1])
def test_one_launch_more_than_the_pipeline(orc, layout):
    """a downscaled submit costs exactly one launch more than an in-place list submit of frames of the downscaled size,
    whatever the source's alignment"""
    import torch

    import h2j_b200 as h2j

    fr = Frames()
    sizes = [(1280, 720), (1279, 719), (640, 360)]
    srcs = [source(orc, w, h, 0, seed=600 + i) for i, (w, h) in enumerate(sizes)]
    y, u, v = downscale_planar(*srcs[0], 2)
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
        for batch in (descs, descs[:1] * 3):  # mixed sizes (list form), one size (batch form)
            l0 = e.kernel_launches
            e.submit_device_downscaled(0, layout, batch, 2)
            assert e.kernel_launches - l0 == l_list + 1
            e.collect(0)
    assert l_list == 7


def test_thumbnail_encoder_and_refusals(orc):
    """an encoder sized for the thumbnail takes 1080p sources at 1/4 and 1/8; what it refuses leaves the previous batch's
    JPEGs and frame info as they were"""
    import torch

    import h2j_b200 as h2j

    fr = Frames()
    y, u, v = source(orc, 1920, 1080, 0, seed=700)
    src = desc(fr, y, u, v, *semiplanar(y, 2048, 8))
    ty, tu, tv = source(orc, 4, 4, 0, seed=701)
    tiny = desc(fr, ty, tu, tv, *planar(ty, tu))
    torch.cuda.synchronize()
    with encoder(0, 2, max_width=480, max_height=272) as e:
        for k in (4, 8):
            e.submit_device_downscaled(0, h2j.LAYOUT_SEMIPLANAR, [src, src], k)
            assert e.collect(0).jpegs == [want_jpeg(orc, y, u, v, k, 0)] * 2
        want4 = orc.oracle_encode(*downscale_planar(y, u, v, 4))
        e.submit_device_downscaled(0, h2j.LAYOUT_SEMIPLANAR, [src], 4)
        info0 = e.frame_info(0, 0)
        d_out, cap, sizes, status = e.collect_device(0)
        assert list(status) == [0] and e.read_device(d_out, int(sizes[0])) == want4[0]

        def refused(layout, descs, k):
            with pytest.raises(h2j.H2JError) as ex:
                e.submit_device_downscaled(0, layout, descs, k)
            info = e.frame_info(0, 0)
            assert (info.qscale, info.scan_bits, info.mcu_w, info.mcu_h) == (info0.qscale, info0.scan_bits, info0.mcu_w, info0.mcu_h)
            assert e.read_device(d_out, int(sizes[0])) == want4[0]
            return ex.value.status

        assert refused(h2j.LAYOUT_SEMIPLANAR, [src], 2) == h2j.ERR_UNSUPPORTED  # 960x540 does not fit 480x272
        for f in (0, 1, 3, 16):
            assert refused(h2j.LAYOUT_SEMIPLANAR, [src], f) == h2j.ERR_INVALID_ARG
        assert refused(h2j.LAYOUT_PLANAR, [tiny], 4) == h2j.ERR_UNSUPPORTED  # 1x1
        assert refused(h2j.LAYOUT_SEMIPLANAR, [src, tiny], 4) == h2j.ERR_INVALID_ARG  # a planar frame's pitches: short pair rows
        assert refused(h2j.LAYOUT_PLANAR, [src, tiny], 4) == h2j.ERR_UNSUPPORTED
        assert refused(h2j.LAYOUT_PLANAR, [], 4) == h2j.ERR_INVALID_ARG
        assert refused(h2j.LAYOUT_PLANAR, [src] * 3, 4) == h2j.ERR_INVALID_ARG  # more than max_batch
        assert refused(2, [src], 4) == h2j.ERR_INVALID_ARG
        big = h2j.FrameDesc(src.data, 65501, 2, 65504, 65504, 65504 * 2, 0)
        assert refused(h2j.LAYOUT_PLANAR, [big], 8) == h2j.ERR_UNSUPPORTED
        e.submit_device_downscaled(0, h2j.LAYOUT_SEMIPLANAR, [src], 8)
        with pytest.raises(h2j.H2JError) as ex:
            e.submit_device_downscaled(0, h2j.LAYOUT_SEMIPLANAR, [src], 8)
        assert ex.value.status == h2j.ERR_BUSY
        assert e.collect(0).jpegs == [want_jpeg(orc, y, u, v, 8, 0)]


def test_full_size_and_thumbnail_from_the_same_surfaces_on_two_slots(orc):
    import torch

    import h2j_b200 as h2j

    fr = Frames()
    n = 4
    srcs = [source(orc, 1920, 1080, 0, "textured" if i % 2 else "noise", 30, seed=800 + i) for i in range(n)]
    descs = [desc(fr, y, u, v, *semiplanar(y, 2048, 8)) for y, u, v in srcs]
    torch.cuda.synchronize()
    with h2j.Encoder(max_width=1920, max_height=1088, max_batch=n, n_slots=2, max_jpeg_bytes=8 * 1024 * 1024) as e:
        e.submit_device_list(0, h2j.LAYOUT_SEMIPLANAR, descs)
        e.submit_device_downscaled(1, h2j.LAYOUT_SEMIPLANAR, descs, 4)
        thumbs = e.collect(1).jpegs
        full = e.collect(0).jpegs
    assert full == [orc.oracle_encode(*p)[0] for p in srcs]
    assert thumbs == [want_jpeg(orc, *p, 4, 0) for p in srcs]


@pytest.mark.parametrize("k", FACTORS)
def test_64_decoder_layout_nv12_frames(orc, k):
    """64 x 1080p NV12 at a hardware decoder's layout (pitch 2048, pair plane behind 1088 rows) in one allocation"""
    import h2j_b200 as h2j

    n, pitch, surf = 64, 2048, 1088
    frame_bytes = pitch * surf * 3 // 2
    bases = [source(orc, 1920, 1080, 0, "textured" if i % 2 else "noise", 20 + 5 * i, seed=900 + i) for i in range(8)]
    rng = random.Random(k)
    pick = [rng.randrange(8) for _ in range(n)]
    placed = [place(y, u, v, *semiplanar(y, pitch, surf - 1080), size=frame_bytes) for y, u, v in bases]
    d, ptr = upload([placed[i] for i in pick], frame_bytes)
    descs = [h2j.FrameDesc(ptr + i * frame_bytes, 1920, 1080, pitch, pitch, pitch * surf, 0) for i in range(n)]
    check = sorted({0, n - 1} | set(rng.sample(range(1, n - 1), 6)))
    w, h = h2j.downscaled_size(1920, 1080, k)
    with h2j.Encoder(max_width=w, max_height=h, max_batch=n, n_slots=1) as e:
        e.submit_device_downscaled(0, h2j.LAYOUT_SEMIPLANAR, descs, k)
        got = e.collect(0).jpegs
    for i in check:
        assert got[i] == want_jpeg(orc, *bases[pick[i]], k, 0), i
