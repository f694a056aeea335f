"""CPU suite: the numpy model of C(frame) (tests/support/rgb.py) that the GPU tests compare the RGB submits with."""
import numpy as np
import pytest

from tests.support import rgb as R

# ITU-T T.871 (JFIF) full-range YCbCr
T871 = {"Y_R": 0.299, "Y_G": 0.587, "Y_B": 0.114, "CB_R": 0.299 / 1.772, "CB_G": 0.587 / 1.772, "CR_G": 0.587 / 1.402, "CR_B": 0.114 / 1.402,
        "HALF": 0.5}


def fix(x):
    return int(x * 65536 + 0.5)


def test_constants_are_fix_of_the_t871_coefficients():
    """jccolor.c writes the coefficients to five decimals; FIX() of those is every constant of the model"""
    for name, c in T871.items():
        assert getattr(R, name) == fix(round(c, 5)), name


@pytest.mark.parametrize("rgb, ycc", [((255, 0, 0), (76, 85, 255)), ((0, 255, 0), (150, 44, 21)), ((0, 0, 255), (29, 255, 107)),
                                      ((255, 255, 255), (255, 128, 128)), ((0, 0, 0), (0, 128, 128)), ((128, 128, 128), (128, 128, 128)),
                                      ((1, 1, 1), (1, 128, 128)), ((254, 254, 254), (254, 128, 128))])
def test_primaries_white_black_and_grey(rgb, ycc):
    assert tuple(R.ycbcr(np.array(rgb, np.uint8))) == ycc


def test_every_triple_is_within_one_of_the_float_formula():
    """over all 2^24 triples: within 1 of T.871 in floating point rounded half up, and different only next to a tie"""
    for r0 in range(0, 256, 32):
        idx = np.arange(32 << 16, dtype=np.int64)
        r, g, b = r0 + (idx >> 16), (idx >> 8) & 255, idx & 255
        got = R.ycbcr(np.stack([r, g, b], -1))
        exact = [0.299 * r + 0.587 * g + 0.114 * b, -T871["CB_R"] * r - T871["CB_G"] * g + 0.5 * b + 128,
                 0.5 * r - T871["CR_G"] * g - T871["CR_B"] * b + 128]
        for k, x in enumerate(exact):
            d = got[:, k] - np.floor(x + 0.5)
            assert np.abs(d).max() <= 1
            assert (got[:, k] >= 0).all() and (got[:, k] <= 255).all()
            assert (np.abs(x[d != 0] - np.floor(x[d != 0]) - 0.5) < 0.01).all(), k


def test_boxes_worked_out_by_hand():
    p = np.array([[10, 11, 12], [20, 21, 22], [31, 32, 40]], np.int64)
    # 2x2: a full box, a 1-wide column, a 1-high row and the 1x1 corner
    assert R.box(p, 2, 2).tolist() == [[(10 + 11 + 20 + 21 + 2) // 4, (12 + 22 + 1) // 2], [(31 + 32 + 1) // 2, 40]]
    # 2x1 (4:2:2): horizontal pairs only, the odd last column alone
    assert R.box(p, 2, 1).tolist() == [[11, 12], [21, 22], [32, 40]]
    assert R.box(np.array([[0, 1]]), 2, 1).tolist() == [[1]]  # (1 + 1) // 2: halves round up
    assert R.box(np.array([[0, 1], [0, 0]]), 2, 2).tolist() == [[0]]  # (1 + 2) // 4
    assert R.box(np.array([[1, 1], [1, 0]]), 2, 2).tolist() == [[1]]  # (3 + 2) // 4
    q = np.random.default_rng(1).integers(0, 256, (7, 9))
    assert (R.box(q, 1, 1) == q).all()  # 4:4:4


@pytest.mark.parametrize("w, h", [(2, 2), (3, 5), (17, 4), (16, 16)])
@pytest.mark.parametrize("cf", [0, 1, 2])
def test_formats_describe_one_picture(w, h, cf):
    """BGR is RGB reversed, X bytes do not matter, planar equals packed; chroma planes have the encoder's sizes"""
    import h2j_b200

    rgb = np.random.default_rng(w * h + cf).integers(0, 256, (h, w, 3), dtype=np.uint8)
    want = R.to_planar(rgb, R.RGB24, cf)
    assert want[1].shape == want[2].shape == h2j_b200.chroma_shape(w, h, cf)
    assert (R.rgb_of(rgb[..., ::-1], R.BGR24) == rgb).all()
    for fmt in R.FORMATS:
        for seed in (0, 1):
            frame = R.as_format(rgb, fmt, seed)
            assert (R.rgb_of(frame, fmt) == rgb).all()
            for a, b in zip(R.to_planar(frame, fmt, cf), want):
                assert (a == b).all(), R.NAMES[fmt]
