"""GPU suite: list batches (h2j_submit_device_list / h2j_submit_host_list), where every frame has its own address and size.
Every JPEG must be byte-identical to the oracle's JPEG of that frame alone.  Device frames sit in separate allocations
surrounded by 0xA5 padding, which must never reach a picture.  Which copy kernels ran is asserted through the encoder's
kernel launch count."""
import random

import numpy as np
import pytest

from tests.test_gpu_formats import CASES

pytestmark = pytest.mark.gpu

PAD = 0xA5
GUARD = 64
BIG_JPEG = 8 * 1024 * 1024


def align(x, a):
    return (x + a - 1) // a * a


def planes(orc, w, h, fmt, kind="textured", seed=0, amp=40):
    return orc.synth_planes_fmt(w, h, fmt, kind, seed=seed, amp=amp)


class Frames:
    """frames in their own device allocations, GUARD bytes of padding on both sides plus `shift` bytes in front"""

    def __init__(self):
        self.keep = []

    def put(self, buf: np.ndarray, shift: int = 0) -> int:
        import torch

        host = np.full(GUARD + shift + buf.size + GUARD, PAD, np.uint8)
        host[GUARD + shift: GUARD + shift + buf.size] = buf
        t = torch.from_numpy(host).cuda()
        self.keep.append(t)
        return t.data_ptr() + GUARD + shift


def planar_desc(h2j, fr, y, u, v, y_pitch=None, c_pitch=None, shift=0):
    h, w = y.shape
    ch, cw = u.shape
    y_pitch = y_pitch or w
    c_pitch = c_pitch or cw
    u_off = y_pitch * h
    v_off = u_off + c_pitch * ch
    buf = np.full(v_off + c_pitch * ch, PAD, np.uint8)
    buf[: y_pitch * h].reshape(h, y_pitch)[:, :w] = y
    buf[u_off: u_off + c_pitch * ch].reshape(ch, c_pitch)[:, :cw] = u
    buf[v_off: v_off + c_pitch * ch].reshape(ch, c_pitch)[:, :cw] = v
    return h2j.FrameDesc(fr.put(buf, shift), w, h, y_pitch, c_pitch, u_off, v_off)


def semiplanar_desc(h2j, fr, y, u, v, pitch, shift=0):
    h, w = y.shape
    ch, cw = u.shape
    uv_off = pitch * h
    buf = np.full(uv_off + pitch * ch, PAD, np.uint8)
    buf[: pitch * h].reshape(h, pitch)[:, :w] = y
    uv = buf[uv_off:].reshape(ch, pitch)
    uv[:, 0: 2 * cw: 2] = u
    uv[:, 1: 2 * cw: 2] = v
    return h2j.FrameDesc(fr.put(buf, shift), w, h, pitch, pitch, uv_off, 0)


def encoder(fmt, max_batch, **kw):
    import h2j_b200

    kw.setdefault("max_jpeg_bytes", BIG_JPEG)
    return h2j_b200.Encoder(max_width=kw.pop("max_width", 1920), max_height=kw.pop("max_height", 1088), max_batch=max_batch, n_slots=1,
                            chroma_format=fmt, **kw)


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
        descs.append(planar_desc(h2j, fr, y, u, v))
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
    descs = [planar_desc(h2j, fr, *f) for f in frames]
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
        descs.append(planar_desc(h2j, fr, y, u, v))
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
        descs.append(planar_desc(h2j, fr, y, u, v, yp, cp, shift))
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
        descs.append(semiplanar_desc(h2j, fr, y, u, v, align(max(w, 2 * u.shape[1]), 64)))
    y, u, v = planes(orc, 131, 77, fmt, seed=89)
    odd = semiplanar_desc(h2j, fr, y, u, v, 2 * u.shape[1] + 3, shift=5)
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
        descs.append(planar_desc(h2j, fr, y, u, v))
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
            descs.append(planar_desc(h2j, fr, *want[(w, h)][1]))
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
        descs.append(planar_desc(h2j, fr, y, u, v))
    limit = max(len(want[0]), len(want[2])) + 16
    assert len(want[1]) > limit
    with encoder(0, len(sizes), max_width=640, max_height=480, max_jpeg_bytes=limit) as e:
        e.submit_device_list(0, h2j.LAYOUT_PLANAR, descs)
        r = e.collect(0, strict=False)
        assert r.status[1] != 0 and r.status[0] == 0 and r.status[2] == 0
        assert r.jpegs[0] == want[0] and r.jpegs[2] == want[2]


def test_argument_errors(orc):
    import h2j_b200 as h2j

    fr = Frames()
    y, u, v = planes(orc, 64, 48, 0)
    good = planar_desc(h2j, fr, y, u, v)
    sp = semiplanar_desc(h2j, fr, y, u, v, 64)

    def with_(d, **kw):
        x = h2j.FrameDesc(d.data, d.width, d.height, d.y_pitch, d.c_pitch, d.u_offset, d.v_offset)
        for k, val in kw.items():
            setattr(x, k, val)
        return x

    with encoder(0, 2, max_width=128, max_height=128) as e:
        def status(layout, descs):
            with pytest.raises(h2j.H2JError) as ex:
                e.submit_device_list(0, layout, descs)
            return ex.value.status

        assert status(h2j.LAYOUT_PLANAR, []) == h2j.ERR_INVALID_ARG
        assert status(h2j.LAYOUT_PLANAR, [good] * 3) == h2j.ERR_INVALID_ARG
        assert status(2, [good]) == h2j.ERR_INVALID_ARG
        assert status(h2j.LAYOUT_PLANAR, [good, with_(good, data=None)]) == h2j.ERR_INVALID_ARG
        assert status(h2j.LAYOUT_PLANAR, [with_(good, y_pitch=63)]) == h2j.ERR_INVALID_ARG
        assert status(h2j.LAYOUT_PLANAR, [with_(good, c_pitch=31)]) == h2j.ERR_INVALID_ARG
        assert status(h2j.LAYOUT_SEMIPLANAR, [with_(sp, c_pitch=63)]) == h2j.ERR_INVALID_ARG
        assert status(h2j.LAYOUT_SEMIPLANAR, [with_(sp, u_offset=64 * 47)]) == h2j.ERR_INVALID_ARG
        assert status(h2j.LAYOUT_PLANAR, [with_(good, width=1)]) == h2j.ERR_UNSUPPORTED
        assert status(h2j.LAYOUT_PLANAR, [with_(good, height=129)]) == h2j.ERR_UNSUPPORTED
        assert status(h2j.LAYOUT_PLANAR, [with_(good, width=70000)]) == h2j.ERR_UNSUPPORTED
        for bad in ([None], None):
            with pytest.raises(h2j.H2JError) as ex:
                if bad is None:
                    e._check(e._lib.h2j_submit_host_list(e._h, 0, None, None, None, 1))
                else:
                    e.submit_host_list(0, [0], [(64, 48)])
            assert ex.value.status == h2j.ERR_INVALID_ARG
        e.submit_device_list(0, h2j.LAYOUT_PLANAR, [good])
        assert status(h2j.LAYOUT_PLANAR, [good]) == h2j.ERR_BUSY
        e.collect(0)


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
    descs = [planar_desc(h2j, fr, *base[s]) for s in sizes]
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
