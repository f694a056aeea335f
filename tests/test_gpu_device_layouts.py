"""GPU suite: device frames at a hardware decoder's layouts (DESIGN.md row (f)(4)) -- semi-planar NV16 / NV24 (and NV12) through
h2j_submit_device_semiplanar, planar frames at any pitches and plane offsets through h2j_submit_device_pitched.  Parity is
defined as for NV12: the JPEG must be byte-identical to the oracle's JPEG of the planar frame with the same samples (and, for
pitched input, to the JPEG of the same frames packed tight through h2j_submit_device).  Padding bytes are 0xA5: they must never
reach the picture.  Which path ran is asserted through the encoder's kernel launch count."""
import pytest

from tests.support.layouts import BIG_JPEG, CASES, align, pipeline_launches, place, run, upload

pytestmark = pytest.mark.gpu


# ---- NV16 / NV24 against the oracle's planar JPEG --------------------------------------------------------------

@pytest.mark.parametrize("layout", ["decoder", "tight", "unaligned"])
@pytest.mark.parametrize("fmt", [1, 2])
def test_semiplanar_matches_planar_split_in_one_launch(orc, fmt, layout):
    import h2j_b200

    with h2j_b200.Encoder(max_width=1920, max_height=1088, max_batch=2, n_slots=1, chroma_format=fmt, max_jpeg_bytes=BIG_JPEG) as e:
        P = pipeline_launches(e)
        for i, (w, h, kind, amp) in enumerate(CASES):
            ch, cw = h2j_b200.chroma_shape(w, h, fmt)
            row = max(w, 2 * cw)
            if layout == "decoder":  # pitch rounded to 256, pair plane behind luma rows padded to a multiple of 16
                pitch, uv_off = align(row, 256), align(row, 256) * align(h, 16)
            else:
                pitch, uv_off = row, row * h
            size = uv_off + pitch * ch
            stride = align(size, 256)
            planes = [orc.synth_planes_fmt(w, h, fmt, kind, seed=300 + 2 * i + s, amp=amp) for s in range(2)]
            want = [orc.oracle_encode(*p, chroma_format=fmt)[0] for p in planes]
            d, ptr = upload([place(*p, pitch, pitch, uv_off, size=size) for p in planes], stride, shift=1 if layout == "unaligned" else 0)
            got, launches = run(e, lambda: e.submit_device_semiplanar(0, ptr, stride, pitch, uv_off, 2, w, h), 2)
            for k in range(2):
                assert got[k] == want[k], f"fmt {fmt} {layout} {w}x{h} frame {k}: JPEG differs from the oracle's planar JPEG"
            in_place = layout != "unaligned" and pitch % 8 == 0 and uv_off % 8 == 0
            expect = P if in_place else P + 1
            assert launches == expect, f"fmt {fmt} {layout} {w}x{h}: {launches} launches, expected {expect} (in place: {in_place})"


@pytest.mark.parametrize("fmt,w,h", [(1, 641, 479), (2, 641, 479), (1, 330, 225), (2, 330, 225), (1, 330, 241), (2, 330, 241),
                                     (1, 2562, 1442), (2, 2562, 1442)])
def test_semiplanar_batches_across_tiles_split_in_one_launch(orc, fmt, w, h):
    """partial tiles, partial units and the predecessor DC across tiles: several tiles per CTA, both paths"""
    import h2j_b200

    n = 4
    ch, cw = h2j_b200.chroma_shape(w, h, fmt)
    pitch = align(max(w, 2 * cw), 256)
    uv_off = pitch * align(h, 16)
    size = uv_off + pitch * ch
    planes = [orc.synth_planes_fmt(w, h, fmt, "textured" if s % 3 else "noise", seed=500 + s, amp=12 + 11 * s) for s in range(n)]
    want = [orc.oracle_encode(*p, chroma_format=fmt)[0] for p in planes]
    d, ptr = upload([place(*p, pitch, pitch, uv_off, size=size) for p in planes], size)
    with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=n, n_slots=1, chroma_format=fmt, max_jpeg_bytes=BIG_JPEG) as e:
        P = pipeline_launches(e)
        for prepass in (0, 1):
            e.set_knob("semiplanar_prepass", prepass)
            for tpc in (0, 2, 5, 16):
                e.set_knob("fdct_tiles_per_cta", tpc)
                got, launches = run(e, lambda: e.submit_device_semiplanar(0, ptr, size, pitch, uv_off, n, w, h), n)
                assert launches == (P + 1 if prepass else P)
                for i in range(n):
                    assert got[i] == want[i], f"fmt {fmt} {w}x{h}, prepass {prepass}, {tpc} tiles per CTA, frame {i}"


@pytest.mark.parametrize("fmt", [1, 2])
def test_semiplanar_range_conversion_and_fixed_qscale(orc, fmt):
    import h2j_b200

    w, h = 322, 242
    ch, cw = h2j_b200.chroma_shape(w, h, fmt)
    pitch = align(2 * cw, 128)
    uv_off = pitch * h
    size = uv_off + pitch * ch
    y, u, v = orc.synth_planes_fmt(w, h, fmt, "textured", seed=77, amp=70)
    d, ptr = upload([place(y, u, v, pitch, pitch, uv_off, size=size)], size)
    for kw in ({"range_mode": 1}, {"fixed_qscale": 3}, {"fixed_qscale": 1}):
        want = orc.oracle_encode(y, u, v, chroma_format=fmt, **kw)[0]
        with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=1, n_slots=1, chroma_format=fmt, max_jpeg_bytes=BIG_JPEG, **kw) as e:
            for prepass in (0, 1):
                e.set_knob("semiplanar_prepass", prepass)
                got, _ = run(e, lambda: e.submit_device_semiplanar(0, ptr, size, pitch, uv_off, 1, w, h), 1)
                assert got[0] == want, (fmt, kw, prepass)


def test_semiplanar_at_420_is_nv12(orc):
    import h2j_b200

    for (w, h, shift, pitch_align) in ((1920, 1080, 0, 256), (330, 241, 0, 8), (17, 9, 1, 1)):
        cw, ch = (w + 1) // 2, (h + 1) // 2
        pitch = align(max(w, 2 * cw), pitch_align)
        uv_off = pitch * h
        size = uv_off + pitch * ch
        stride = align(size, 256)
        planes = [orc.synth_planes(w, h, "textured", seed=90 + s) for s in range(2)]
        d, ptr = upload([place(*p, pitch, pitch, uv_off, size=size) for p in planes], stride, shift)
        with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=2, n_slots=1) as e:
            a, la = run(e, lambda: e.submit_device_nv12(0, ptr, stride, pitch, uv_off, 2, w, h), 2)
            b, lb = run(e, lambda: e.submit_device_semiplanar(0, ptr, stride, pitch, uv_off, 2, w, h), 2)
        assert a == b and la == lb, (w, h)
        assert a == [orc.oracle_encode(*p)[0] for p in planes], (w, h)


# ---- planar frames at any layout ------------------------------------------------------------------------------

def pitched_layouts(w, h, fmt):
    """name -> (y_pitch, c_pitch, u_off, v_off, size, base shift)"""
    import h2j_b200

    ch, cw = h2j_b200.chroma_shape(w, h, fmt)
    out = {}
    p, sh = align(w, 256), align(h, 16)  # a decoder surface: one pitch, planes at multiples of pitch * surface height
    out["nvdec"] = (p, p, p * sh, 2 * p * sh, 2 * p * sh + p * ch, 0)
    y_sz = w * h  # YV12 order: V in front of U, tight rows
    out["yv12"] = (w, cw, y_sz + cw * ch, y_sz, y_sz + 2 * cw * ch, 0)
    yp, cp = align(w, 64), align(cw, 32) + 8  # luma and chroma pitches differ
    u0 = yp * h + 40
    out["two_pitches"] = (yp, cp, u0, u0 + cp * ch + 24, u0 + 2 * cp * ch + 24, 0)
    out["unaligned"] = out["nvdec"][:5] + (3,)
    return out


@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_pitched_matches_tight_planar(orc, fmt):
    import h2j_b200

    for (w, h) in ((1920, 1080), (641, 479), (33, 17)):
        n = 2
        planes = [orc.synth_planes_fmt(w, h, fmt, "textured", seed=700 + s, amp=30 + 20 * s) for s in range(n)]
        tight = [orc.pack_i420(*p) for p in planes]
        tstride = align(len(tight[0]), 256)
        with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=n, n_slots=1, chroma_format=fmt, max_jpeg_bytes=BIG_JPEG) as e:
            P = pipeline_launches(e)
            dt, tptr = upload(tight, tstride)
            want, _ = run(e, lambda: e.submit_device(0, tptr, tstride, n, w, h), n)
            assert want == [orc.oracle_encode(*p, chroma_format=fmt)[0] for p in planes]
            for name, (yp, cp, uo, vo, size, shift) in pitched_layouts(w, h, fmt).items():
                stride = align(size, 256)
                d, ptr = upload([place(*p, yp, cp, uo, vo, size) for p in planes], stride, shift)
                got, launches = run(e, lambda: e.submit_device_pitched(0, ptr, stride, yp, cp, uo, vo, n, w, h), n)
                assert got == want, f"fmt {fmt} {w}x{h} {name}"
                aligned = shift % 8 == 0 and all(x % 8 == 0 for x in (yp, cp, uo, vo, stride))
                assert launches == (P if aligned else P + 1), f"fmt {fmt} {w}x{h} {name}: {launches} launches"
