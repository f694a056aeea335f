"""Exact numpy model of C(frame), the planar frame h2j_submit_device_rgb and h2j_encode_frame_rgb encode for an RGB frame
(include/h2j_b200.h): per pixel JFIF / T.871 full-range YCbCr in libjpeg's 16-bit fixed point, then the Cb and Cr planes
box-averaged to the chroma format's sizes, (S + c/2) // c over the c samples of a box that lie inside the plane; and the
RGB device frames the GPU tests submit."""
import numpy as np
from numpy.lib.stride_tricks import as_strided

from tests.support.layouts import PAD

RGB24, BGR24, RGBX, BGRX, PLANAR = range(5)
FORMATS = (RGB24, BGR24, RGBX, BGRX, PLANAR)
NAMES = {RGB24: "RGB24", BGR24: "BGR24", RGBX: "RGBX", BGRX: "BGRX", PLANAR: "planar"}
BYTES_PER_PIXEL = {RGB24: 3, BGR24: 3, RGBX: 4, BGRX: 4, PLANAR: 1}

# jccolor.c's fixed-point constants: FIX(x) = (int)(x * 65536 + 0.5)
Y_R, Y_G, Y_B = 19595, 38470, 7471
CB_R, CB_G = 11059, 21709
CR_G, CR_B = 27439, 5329
HALF = 32768  # FIX(0.5): the B term of Cb and the R term of Cr
BOX = {0: (2, 2), 1: (2, 1), 2: (1, 1)}  # chroma format -> (kx, ky)


def ycbcr(rgb: np.ndarray) -> np.ndarray:
    """(..., 3) R, G, B -> (..., 3) int64 Y, Cb, Cr"""
    r, g, b = (rgb[..., i].astype(np.int64) for i in range(3))
    y = (Y_R * r + Y_G * g + Y_B * b + 32768) >> 16
    cb = (-CB_R * r - CB_G * g + HALF * b + (128 << 16) + 32767) >> 16
    cr = (HALF * r - CR_G * g - CR_B * b + (128 << 16) + 32767) >> 16
    return np.stack([y, cb, cr], -1)


def box(plane: np.ndarray, kx: int, ky: int) -> np.ndarray:
    """kx x ky box averages of a 2-D plane, rounded half up over the samples of each box inside the plane"""
    ph, pw = plane.shape
    oh, ow = -(-ph // ky), -(-pw // kx)
    pad = np.zeros((oh * ky, ow * kx), np.int64)
    pad[:ph, :pw] = plane
    ones = np.zeros((oh * ky, ow * kx), np.int64)
    ones[:ph, :pw] = 1
    s = pad.reshape(oh, ky, ow, kx).sum(axis=(1, 3))
    c = ones.reshape(oh, ky, ow, kx).sum(axis=(1, 3))
    return ((s + c // 2) // c).astype(np.uint8)


def rgb_of(frame: np.ndarray, fmt: int) -> np.ndarray:
    """a frame of format fmt ((H, W, 3|4) packed, (3, H, W) planar) -> its (H, W, 3) R, G, B picture"""
    if fmt == PLANAR:
        return frame.transpose(1, 2, 0)
    return frame[..., 2::-1] if fmt in (BGR24, BGRX) else frame[..., :3]


def as_format(rgb: np.ndarray, fmt: int, seed: int = 0) -> np.ndarray:
    """an (H, W, 3) R, G, B picture as a frame of format fmt; X bytes are random"""
    if fmt == PLANAR:
        return np.ascontiguousarray(rgb.transpose(2, 0, 1))
    px = rgb[..., ::-1] if fmt in (BGR24, BGRX) else rgb
    if fmt in (RGBX, BGRX):
        x = np.random.default_rng(seed).integers(0, 256, rgb.shape[:2] + (1,), dtype=np.uint8)
        px = np.concatenate([px, x], -1)
    return np.ascontiguousarray(px)


def to_planar(frame: np.ndarray, fmt: int, chroma_format: int):
    """C(frame): (y, u, v) uint8 planes at the chroma format"""
    ycc = ycbcr(rgb_of(frame, fmt))
    kx, ky = BOX[chroma_format]
    return ycc[..., 0].astype(np.uint8), box(ycc[..., 1], kx, ky), box(ycc[..., 2], kx, ky)


def place_rgb(fr, frame: np.ndarray, fmt: int, pitch: int = None, shift: int = 0, gap: int = 0):
    """the h2j_b200.FrameDesc of a frame put by fr (tests/support/layouts.Frames) into its own allocation, `shift` bytes past
    an aligned start: rows `pitch` bytes apart (default: tight), planar planes each followed by `gap` spare rows; every
    byte between is PAD"""
    import h2j_b200

    if fmt == PLANAR:
        _, h, w = frame.shape
        rows = [p for p in frame]
    else:
        h, w = frame.shape[:2]
        rows = [frame.reshape(h, -1)]
    row = rows[0].shape[1]
    pitch = pitch or row
    plane = pitch * (h + gap)
    buf = np.full(plane * (len(rows) - 1) + pitch * (h - 1) + row, PAD, np.uint8)
    for k, p in enumerate(rows):
        as_strided(buf[k * plane:], shape=p.shape, strides=(pitch, 1))[:] = p
    data = fr.put(buf, shift)
    planar = fmt == PLANAR
    return h2j_b200.FrameDesc(data, w, h, pitch, 0, plane if planar else 0, 2 * plane if planar else 0)
