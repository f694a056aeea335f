"""GPU suite: list batches (h2j_submit_device_list / h2j_submit_host_list), where every frame has its own address and size.
Every JPEG must be byte-identical to the oracle's JPEG of that frame alone.  Device frames sit in separate allocations
surrounded by 0xA5 padding, which must never reach a picture.  Which copy kernels ran is asserted through the encoder's
kernel launch count."""
import random

import numpy as np
import pytest

from tests.support.layouts import CASES, Frames, align, desc, encoder, planar, semiplanar

pytestmark = pytest.mark.gpu


def planes(orc, w, h, fmt, kind="textured", seed=0, amp=40):
    return orc.synth_planes_fmt(w, h, fmt, kind, seed=seed, amp=amp)


def collect_jpegs(e, n):
    r = e.collect(0)
    return list(r.jpegs[:n])


@pytest.mark.parametrize("fmt", [0, 1, 2])
@pytest.mark.parametrize("order", ["ascending", "descending", "shuffled"])
def test_all_sizes_in_one_batch(orc, fmt, order):
    import h2j_b200 as h2j

    cases = sorted(CASES, key=lambda c: c[0] * c[1])
    if order == "descending":
        cases = cases[::-1]
    elif order == "shuffled":
        random.Random(7).shuffle(cases)
    fr = Frames()
    descs, want = [], []
    for i, (w, h, kind, amp) in enumerate(cases):
        y, u, v = planes(orc, w, h, fmt, kind, seed=30 + i, amp=amp)
        want.append(orc.oracle_encode(y, u, v, chroma_format=fmt)[0])
        descs.append(desc(fr, y, u, v, *planar(y, u)))
    with encoder(fmt, len(cases)) as e:
        e.submit_device_list(0, h2j.LAYOUT_PLANAR, descs)
        got = collect_jpegs(e, len(cases))
    for (w, h, _, _), g, wnt in zip(cases, got, want):
        assert g == wnt, f"{w}x{h} fmt {fmt} {order}"


@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_uniform_list_equals_submit_device(orc, fmt):
    import torch

    import h2j_b200 as h2j

    w, h, n = 641, 479, 5
    frames = [planes(orc, w, h, fmt, "noise", seed=50 + i, amp=20) for i in range(n)]
    tight = np.concatenate([np.concatenate([p.ravel() for p in f]) for f in frames])
    fb = tight.size // n
    fr = Frames()
    descs = [desc(fr, y, u, v, *planar(y, u)) for y, u, v in frames]
    with encoder(fmt, n) as e:
        d = torch.from_numpy(tight).cuda()
        e.submit_device(0, d.data_ptr(), fb, n, w, h)
        infos_a = [e.frame_info(0, i) for i in range(n)]
        a = collect_jpegs(e, n)
        e.submit_device_list(0, h2j.LAYOUT_PLANAR, descs)
        infos_b = [e.frame_info(0, i) for i in range(n)]
        b = collect_jpegs(e, n)
    assert a == b
    for x, y in zip(infos_a, infos_b):
        assert (x.qscale, x.mb_var_sum, x.mcu_w, x.mcu_h, x.header_bytes, x.scan_bits) == (y.qscale, y.mb_var_sum, y.mcu_w, y.mcu_h, y.header_bytes, y.scan_bits)


def test_frame_info_and_coefficients_answer_for_the_frame(orc):
    import h2j_b200 as h2j

    sizes = [(1280, 720), (33, 47), (641, 479)]
    fr = Frames()
    descs, dbgs = [], []
    for i, (w, h) in enumerate(sizes):
        y, u, v = planes(orc, w, h, 0, seed=60 + i)
        _, dbg, coefs = orc.oracle_encode(y, u, v, want_coefs=True)
        dbgs.append((dbg, coefs))
        descs.append(desc(fr, y, u, v, *planar(y, u)))
    with encoder(0, len(sizes)) as e:
        e.submit_device_list(0, h2j.LAYOUT_PLANAR, descs)
        for i, (dbg, coefs) in enumerate(dbgs):
            info = e.frame_info(0, i)
            assert (info.mcu_w, info.mcu_h) == (dbg.mcu_w, dbg.mcu_h)
            assert (e.coefficients(0, i, coefs.shape[0]) == coefs).all()
        e.collect(0)


@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_pitched_aligned_and_unaligned_mixed(orc, fmt):
    import h2j_b200 as h2j

    specs = [(1920, 1080, 2048, None, 0), (1918, 1078, None, None, 0), (641, 479, 704, 704 if fmt == 2 else 384, 0), (322, 242, None, None, 3),
             (1280, 720, 1280, 640 if fmt != 2 else 1280, 0), (17, 17, None, None, 1)]
    fr = Frames()
    descs, want = [], []
    for i, (w, h, yp, cp, shift) in enumerate(specs):
        y, u, v = planes(orc, w, h, fmt, seed=70 + i)
        want.append(orc.oracle_encode(y, u, v, chroma_format=fmt)[0])
        y_pitch, c_pitch, u_off, v_off = planar(y, u, yp, cp)
        descs.append(desc(fr, y, u, v, y_pitch, c_pitch, u_off, v_off, size=v_off + c_pitch * u.shape[0], shift=shift))
    aligned = [d for d, s in zip(descs, specs) if s[0] in (1920, 1280) or s[2] == 704]
    with encoder(fmt, len(specs)) as e:
        l0 = e.kernel_launches
        e.submit_device_list(0, h2j.LAYOUT_PLANAR, aligned)
        l_plain = e.kernel_launches - l0
        collect_jpegs(e, len(aligned))
        l0 = e.kernel_launches
        e.submit_device_list(0, h2j.LAYOUT_PLANAR, descs)
        assert e.kernel_launches - l0 == l_plain + 1, "the unaligned frames are copied in exactly one launch"
        got = collect_jpegs(e, len(specs))
    assert l_plain == 7  # K1 .. K5 and the offsets kernel: no copy for an all-aligned batch
    assert got == want


@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_semiplanar_in_place_and_split(orc, fmt):
    import h2j_b200 as h2j

    sizes = [(1920, 1080), (1280, 720), (641, 479), (64, 64), (17, 17)]
    fr = Frames()
    descs, want = [], []
    for i, (w, h) in enumerate(sizes):
        y, u, v = planes(orc, w, h, fmt, seed=80 + i)
        want.append(orc.oracle_encode(y, u, v, chroma_format=fmt)[0])
        pitch = align(max(w, 2 * u.shape[1]), 64)
        descs.append(desc(fr, y, u, v, *semiplanar(y, pitch), size=pitch * (h + u.shape[0])))
    y, u, v = planes(orc, 131, 77, fmt, seed=89)
    pitch = 2 * u.shape[1] + 3
    odd = desc(fr, y, u, v, *semiplanar(y, pitch), size=pitch * (77 + u.shape[0]), shift=5)
    want_odd = orc.oracle_encode(y, u, v, chroma_format=fmt)[0]
    with encoder(fmt, len(sizes) + 1) as e:
        l0 = e.kernel_launches
        e.submit_device_list(0, h2j.LAYOUT_SEMIPLANAR, descs)
        l_in_place = e.kernel_launches - l0
        assert collect_jpegs(e, len(sizes)) == want
        l0 = e.kernel_launches
        e.submit_device_list(0, h2j.LAYOUT_SEMIPLANAR, descs[:2] + [odd] + descs[2:])
        assert e.kernel_launches - l0 == l_in_place + 1
        assert collect_jpegs(e, len(sizes) + 1) == want[:2] + [want_odd] + want[2:]
    assert l_in_place == 7


@pytest.mark.parametrize("tiles", [2, 5, 16])
@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_several_tiles_per_cta(orc, fmt, tiles):
    import h2j_b200 as h2j

    sizes = [(641, 479), (330, 241), (17, 4098), (2562, 1442)]
    fr = Frames()
    descs, want = [], []
    for i, (w, h) in enumerate(sizes):
        y, u, v = planes(orc, w, h, fmt, "noise", seed=90 + i, amp=30)
        want.append(orc.oracle_encode(y, u, v, chroma_format=fmt)[0])
        descs.append(desc(fr, y, u, v, *planar(y, u)))
    with encoder(fmt, len(sizes), max_width=2562, max_height=4098) as e:
        e.set_knob("fdct_tiles_per_cta", tiles)
        e.submit_device_list(0, h2j.LAYOUT_PLANAR, descs)
        assert collect_jpegs(e, len(sizes)) == want


def test_both_scan_place_widths(orc):
    """a small batch has fewer K4b groups than two per SM (the 8-units-per-warp form), a large one more (the 32 form): its
    largest frame is 1080p, six groups of 256 units, so 64 frames launch 384 groups, above 2 x 148 SMs"""
    import h2j_b200 as h2j

    small = [(64, 64), (131, 77)]
    large = [(1920, 1080), (1280, 720)] * 32
    for sizes in (small, large):
        fr = Frames()
        descs, want = [], {}
        for i, (w, h) in enumerate(sizes):
            if (w, h) not in want:
                y, u, v = planes(orc, w, h, 0, seed=100 + len(want))
                want[(w, h)] = (orc.oracle_encode(y, u, v)[0], (y, u, v))
            y, u, v = want[(w, h)][1]
            descs.append(desc(fr, y, u, v, *planar(y, u)))
        with encoder(0, len(sizes)) as e:
            e.set_profile(True)
            e.submit_device_list(0, h2j.LAYOUT_PLANAR, descs)
            got = collect_jpegs(e, len(sizes))
        assert got == [want[s][0] for s in sizes]


def test_one_frame_over_the_limit_fails_alone(orc):
    import h2j_b200 as h2j

    sizes = [(322, 242, "textured", 40), (640, 480, "noise", 100), (64, 64, "textured", 40)]
    fr = Frames()
    descs, want = [], []
    for i, (w, h, kind, amp) in enumerate(sizes):
        y, u, v = planes(orc, w, h, 0, kind, seed=110 + i, amp=amp)
        want.append(orc.oracle_encode(y, u, v)[0])
        descs.append(desc(fr, y, u, v, *planar(y, u)))
    limit = max(len(want[0]), len(want[2])) + 16
    assert len(want[1]) > limit
    with encoder(0, len(sizes), max_width=640, max_height=480, max_jpeg_bytes=limit) as e:
        e.submit_device_list(0, h2j.LAYOUT_PLANAR, descs)
        r = e.collect(0, strict=False)
        assert r.status[1] != 0 and r.status[0] == 0 and r.status[2] == 0
        assert r.jpegs[0] == want[0] and r.jpegs[2] == want[2]


def test_large_mixed_batch(orc):
    import h2j_b200 as h2j

    kinds = [(3840, 2160), (1920, 1080), (1280, 720)]
    rng = random.Random(3)
    sizes = [kinds[rng.randrange(3)] for _ in range(256)]
    base = {}
    for i, s in enumerate(kinds):
        y, u, v = planes(orc, *s, 0, seed=120 + i)
        base[s] = (y, u, v)
    fr = Frames()
    descs = [desc(fr, y, u, v, *planar(y, u)) for y, u, v in (base[s] for s in sizes)]
    check = sorted({0, 255} | set(rng.sample(range(256), 6)))
    with encoder(0, 256, max_width=3840, max_height=2160) as e:
        e.submit_device_list(0, h2j.LAYOUT_PLANAR, descs)
        got = collect_jpegs(e, 256)
    for i in check:
        assert got[i] == orc.oracle_encode(*base[sizes[i]])[0], i


@pytest.mark.parametrize("pinned", [False, True])
def test_host_list(orc, pinned):
    import h2j_b200 as h2j

    sizes = [(1920, 1080), (17, 17), (641, 479), (1918, 1078), (2, 2)]
    frames, want, keep = [], [], []
    for i, (w, h) in enumerate(sizes):
        y, u, v = planes(orc, w, h, 0, seed=130 + i)
        want.append(orc.oracle_encode(y, u, v)[0])
        tight = np.concatenate([y.ravel(), u.ravel(), v.ravel()])
        if pinned:
            buf = h2j.PinnedBuffer(tight.size)
            np.ctypeslib.as_array((np.ctypeslib.ctypes.c_uint8 * tight.size).from_address(buf.ptr))[:] = tight
            keep.append(buf)
            frames.append(buf.ptr)
        else:
            keep.append(tight)
            frames.append(tight.ctypes.data)
    with encoder(0, len(sizes)) as e:
        e.submit_host_list(0, frames, sizes)
        assert collect_jpegs(e, len(sizes)) == want
