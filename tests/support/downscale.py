"""Exact numpy model of the box filter D_k that h2j_submit_device_downscaled applies (include/h2j_b200.h): every plane at its
decoder size pw x ph becomes ceil(pw/k) x ceil(ph/k), out[y][x] = (S + c/2) // c over the c samples of the box that lie
inside the plane (int64 sums), semi-planar Cb and Cr separately."""
import numpy as np

FACTORS = (2, 4, 8)


def downscaled_shape(rows: int, cols: int, k: int):
    return -(-rows // k), -(-cols // k)


def box_plane(p: np.ndarray, k: int) -> np.ndarray:
    """one plane (2-D uint8) -> its k-box averages, rounded half up"""
    assert k in FACTORS and p.ndim == 2
    ph, pw = p.shape
    oh, ow = downscaled_shape(ph, pw, k)
    pad = np.zeros((oh * k, ow * k), np.int64)
    pad[:ph, :pw] = p
    ones = np.zeros((oh * k, ow * k), np.int64)
    ones[:ph, :pw] = 1
    s = pad.reshape(oh, k, ow, k).sum(axis=(1, 3))
    c = ones.reshape(oh, k, ow, k).sum(axis=(1, 3))
    return ((s + c // 2) // c).astype(np.uint8)


def downscale_planar(y: np.ndarray, u: np.ndarray, v: np.ndarray, k: int):
    """D_k of a planar frame: (y, u, v) of the downscaled frame"""
    return box_plane(y, k), box_plane(u, k), box_plane(v, k)


def downscale_semiplanar(y: np.ndarray, uv: np.ndarray, k: int):
    """D_k of a semi-planar frame (uv: rows of interleaved Cb/Cr pairs, 2 * pairs wide): the downscaled PLANAR frame"""
    assert uv.ndim == 2 and uv.shape[1] % 2 == 0
    return box_plane(y, k), box_plane(uv[:, 0::2], k), box_plane(uv[:, 1::2], k)
