"""CPU suite: the numpy model of D_k (tests/support/downscale.py) on boxes worked out by hand, and the chroma-size identity
that lets a downscaled frame keep its format's chroma planes: ceil(ceil(w/2)/k) == ceil(ceil(w/k)/2)."""
import numpy as np
import pytest

from tests.support.downscale import FACTORS, box_plane, downscale_planar, downscale_semiplanar, downscaled_shape


def test_3x3_at_2_full_partial_and_corner_boxes():
    p = np.array([[10, 20, 30],
                  [40, 50, 60],
                  [70, 80, 91]], np.uint8)
    got = box_plane(p, 2)
    assert got.shape == (2, 2)
    assert got[0, 0] == (10 + 20 + 40 + 50 + 2) // 4  # full box: 30
    assert got[0, 1] == (30 + 60 + 1) // 2            # column-partial: 45
    assert got[1, 0] == (70 + 80 + 1) // 2            # row-partial: 75
    assert got[1, 1] == 91                            # corner: one sample
    assert got.tolist() == [[30, 45], [75, 91]]


@pytest.mark.parametrize("samples,want", [([1, 2], 2), ([0, 0, 0, 1], 0), ([0, 0, 1, 1], 1), ([1, 2, 2], 2)])
def test_rounding_half_up(samples, want):
    if len(samples) == 2:  # a column-partial box: 1 x 2 of a 2-row, 1-column plane
        p = np.array(samples, np.uint8).reshape(2, 1)
    elif len(samples) == 4:
        p = np.array(samples, np.uint8).reshape(2, 2)
    else:  # three samples: the row-partial edge box of a 4 x 3 plane at k = 4 (one row of three)
        p = np.array([samples], np.uint8)
        assert box_plane(p, 4).shape == (1, 1)
        assert box_plane(p, 4)[0, 0] == want
        return
    assert box_plane(p, 2)[0, 0] == want


def test_three_sample_edge_box_inside_a_larger_plane():
    p = np.zeros((3, 3), np.uint8)
    p[2, 0], p[2, 1] = 1, 2  # bottom row-partial box of (1, 2) and ...
    p[0, 2], p[1, 2] = 2, 2
    got = box_plane(p, 2)
    assert got[1, 0] == 2  # (1 + 2 + 1) // 2
    assert got[0, 1] == 2


@pytest.mark.parametrize("k", FACTORS)
@pytest.mark.parametrize("pw,ph", [(1, 1), (1, 5), (3, 2), (7, 9)])
def test_planes_narrower_than_k(k, pw, ph):
    rng = np.random.default_rng(pw * 100 + ph + k)
    p = rng.integers(0, 256, (ph, pw)).astype(np.uint8)
    got = box_plane(p, k)
    assert got.shape == downscaled_shape(ph, pw, k)
    for oy in range(got.shape[0]):
        for ox in range(got.shape[1]):
            box = p[oy * k: oy * k + k, ox * k: ox * k + k].astype(np.int64)
            assert got[oy, ox] == (box.sum() + box.size // 2) // box.size


@pytest.mark.parametrize("k", FACTORS)
def test_model_against_a_loop(k):
    rng = np.random.default_rng(k)
    p = rng.integers(0, 256, (37, 53)).astype(np.uint8)
    got = box_plane(p, k)
    for oy in range(got.shape[0]):
        for ox in range(got.shape[1]):
            box = [int(p[j, i]) for j in range(oy * k, min(oy * k + k, 37)) for i in range(ox * k, min(ox * k + k, 53))]
            assert got[oy, ox] == (sum(box) + len(box) // 2) // len(box)
    assert box_plane(np.full((16, 16), 255, np.uint8), k).min() == 255


def test_semiplanar_averages_cb_and_cr_separately():
    y = np.zeros((4, 4), np.uint8)
    uv = np.array([[10, 200, 20, 100], [30, 0, 40, 255]], np.uint8)  # 2 rows of 2 pairs
    _, u, v = downscale_semiplanar(y, uv, 2)
    assert u.tolist() == [[25]] and v.tolist() == [[(200 + 100 + 0 + 255 + 2) // 4]]
    _, u2, v2 = downscale_planar(y, uv[:, 0::2].copy(), uv[:, 1::2].copy(), 2)
    assert (u == u2).all() and (v == v2).all()


@pytest.mark.parametrize("k", FACTORS)
@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_chroma_size_identity(fmt, k):
    """the downscaled chroma planes are the downscaled frame's chroma planes, for every width and height below 3000"""
    from h2j_b200 import chroma_shape, downscaled_size

    for s in range(2, 3000):
        dw, dh = downscaled_size(s, s, k)
        ch, cw = chroma_shape(s, s, fmt)
        assert downscaled_shape(ch, cw, k) == chroma_shape(dw, dh, fmt), (fmt, k, s)


def test_downscaled_size_refuses_other_factors():
    from h2j_b200 import downscaled_size

    assert downscaled_size(1920, 1080, 4) == (480, 270)
    assert downscaled_size(17, 4098, 8) == (3, 513)
    for f in (0, 1, 3, 16):
        with pytest.raises(ValueError):
            downscaled_size(64, 64, f)
