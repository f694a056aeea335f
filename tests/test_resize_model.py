"""CPU suite: the numpy model of R(frame) (tests/support/resize.py) against PIL.Image.resize itself, for BOX, BILINEAR and
BICUBIC, on a seeded sweep of size pairs (down, up, one axis or none changed, 2 on a side, odd sizes, the ratios services
ask for) and on contents that drive bicubic's clipping at both ends; and the chroma sizes of a resized frame."""
import numpy as np
import pytest

from tests.support.resize import FILTERS, coeffs, resize_plane, resize_planar, resize_semiplanar

Image = pytest.importorskip("PIL.Image")
PIL_FILTER = {0: Image.BOX, 1: Image.BILINEAR, 2: Image.BICUBIC}


def content(rng, h, w, kind):
    if kind == "random":
        return rng.integers(0, 256, (h, w), dtype=np.uint8)
    if kind == "gradient":
        return ((np.arange(w)[None, :] * 7 + np.arange(h)[:, None] * 3) % 256).astype(np.uint8)
    if kind == "steps":  # 0/255 steps every few samples: overshoot above 255 and below 0
        return np.where((np.arange(w)[None, :] // 3 + np.arange(h)[:, None] // 2) % 2 == 0, 255, 0).astype(np.uint8)
    return np.where((np.arange(w)[None, :] + np.arange(h)[:, None]) % 2 == 0, 255, 0).astype(np.uint8)  # checkerboard


def size_pairs():
    """((w, h), (W, H)): named cases, then a seeded sweep"""
    named = [((2, 2), (2, 2)), ((2, 2), (7, 3)), ((9, 5), (2, 2)), ((2, 9), (2, 3)), ((300, 2), (17, 2)),
             ((1920, 1080), (1280, 720)), ((1920, 1080), (640, 360)), ((1920, 1080), (320, 180)), ((1080, 1080), (224, 224)),
             ((1920, 1080), (224, 224)), ((854, 480), (1280, 720)), ((33, 47), (33, 20)), ((33, 47), (50, 47)), ((33, 47), (33, 47)),
             ((481, 271), (160, 90)), ((99, 77), (396, 77)), ((640, 360), (512, 288))]
    rng = np.random.default_rng(2026)
    sweep = []
    for i in range(400):
        w, h = (int(x) for x in rng.integers(2, 300, 2))
        if i % 4 == 0:
            W, H = max(2, w // int(rng.integers(1, 9))), max(2, h // int(rng.integers(1, 9)))
        elif i % 4 == 1:
            W, H = (int(x) for x in rng.integers(2, 600, 2))
        elif i % 4 == 2:
            W, H = (w, int(rng.integers(2, 300))) if i % 8 == 2 else (int(rng.integers(2, 300)), h)
        else:
            W, H = (int(x) for x in rng.integers(2, 300, 2))
        sweep.append(((w, h), (W, H)))
    return named + sweep


KINDS = ("random", "gradient", "steps", "checker")


@pytest.mark.parametrize("flt", FILTERS)
def test_model_equals_pillow_on_a_sweep(flt):
    rng = np.random.default_rng(flt)
    for i, ((w, h), (W, H)) in enumerate(size_pairs()):
        p = content(rng, h, w, KINDS[i % 4])
        want = np.asarray(Image.fromarray(p, "L").resize((W, H), PIL_FILTER[flt]))
        got = resize_plane(p, W, H, flt)
        assert got.shape == (H, W) and np.array_equal(got, want), ((w, h), (W, H), flt, KINDS[i % 4])


@pytest.mark.parametrize("flt", FILTERS)
@pytest.mark.parametrize("kind", KINDS)
def test_one_very_long_axis(flt, kind):
    rng = np.random.default_rng(7)
    for (w, h), (W, H) in (((20000, 3), (7, 3)), ((3, 20000), (3, 7)), ((5, 3), (20000, 3))):
        p = content(rng, h, w, kind)
        want = np.asarray(Image.fromarray(p, "L").resize((W, H), PIL_FILTER[flt]))
        assert np.array_equal(resize_plane(p, W, H, flt), want), ((w, h), (W, H))


def test_bicubic_clips_at_both_ends():
    p = content(None, 6, 40, "steps")
    raw_min = raw_max = 0
    xmin, n, k = coeffs(40, 97, 2)
    for o in range(97):  # the unclipped horizontal sums of row 0 overshoot both ends
        s = (1 << 21) + int((p[0, xmin[o]: xmin[o] + n[o]].astype(np.int64) * k[o, : n[o]]).sum())
        raw_min, raw_max = min(raw_min, s >> 22), max(raw_max, s >> 22)
    assert raw_min < 0 and raw_max > 255
    assert np.array_equal(resize_plane(p, 97, 6, 2), np.asarray(Image.fromarray(p, "L").resize((97, 6), Image.BICUBIC)))


def test_identity_and_box_is_not_the_integer_box_average():
    rng = np.random.default_rng(3)
    p = rng.integers(0, 256, (31, 45), dtype=np.uint8)
    for flt in FILTERS:
        assert np.array_equal(resize_plane(p, 45, 31, flt), p)
    # Pillow's BOX at 1/2 rounds between its passes: it differs from the rounded 2x2 average on some samples
    from tests.support.downscale import box_plane

    q = rng.integers(0, 256, (64, 64), dtype=np.uint8)
    assert not np.array_equal(resize_plane(q, 32, 32, 0), box_plane(q, 2))


@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_chroma_planes_take_the_output_frames_chroma_size(fmt):
    from h2j_b200 import chroma_shape

    rng = np.random.default_rng(fmt)
    for (w, h), (W, H) in (((17, 9), (6, 31)), ((1920, 1080), (224, 224)), ((2, 2), (3, 3)), ((101, 55), (101, 55))):
        ch, cw = chroma_shape(w, h, fmt)
        y = rng.integers(0, 256, (h, w), dtype=np.uint8)
        u = rng.integers(0, 256, (ch, cw), dtype=np.uint8)
        v = rng.integers(0, 256, (ch, cw), dtype=np.uint8)
        ry, ru, rv = resize_planar(y, u, v, W, H, fmt, 1)
        assert ry.shape == (H, W) and ru.shape == rv.shape == chroma_shape(W, H, fmt)
        for plane, got in ((u, ru), (v, rv)):
            want = Image.fromarray(plane, "L").resize((got.shape[1], got.shape[0]), Image.BILINEAR)
            assert np.array_equal(got, np.asarray(want))
        uv = np.empty((ch, 2 * cw), np.uint8)
        uv[:, 0::2], uv[:, 1::2] = u, v
        assert all(np.array_equal(a, b) for a, b in zip(resize_semiplanar(y, uv, W, H, fmt, 1), (ry, ru, rv)))
    assert chroma_shape(225, 223, fmt) == {0: (112, 113), 1: (223, 113), 2: (223, 225)}[fmt]
