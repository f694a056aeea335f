"""Exact numpy model of R(frame), the resized frame h2j_submit_device_resized encodes (include/h2j_b200.h): every plane
resized as a Pillow "L" image by PIL.Image.resize with BOX, BILINEAR or BICUBIC (libImaging/Resample.c).  The coefficients
are built with Python floats (IEEE double) in Pillow's order of operations; the passes are integer sums, vectorised over
rows.  tests/test_resize_model.py pins this against Pillow itself."""
import numpy as np

BOX, BILINEAR, BICUBIC = 0, 1, 2  # h2j_b200.FILTER_*
FILTERS = (BOX, BILINEAR, BICUBIC)
PRECISION_BITS = 22
SUPPORT = {BOX: 0.5, BILINEAR: 1.0, BICUBIC: 2.0}


def _filter(flt, x):
    if flt == BOX:
        return 1.0 if -0.5 < x <= 0.5 else 0.0
    x = abs(x)
    if flt == BILINEAR:
        return 1.0 - x if x < 1.0 else 0.0
    a = -0.5
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0:
        return (((x - 5) * x + 8) * x - 4) * a
    return 0.0


def coeffs(n_in: int, n_out: int, flt: int):
    """(xmin[out], n[out], k[out][ksize]) of one axis: Pillow's precompute_coeffs + normalize_coeffs_8bpc (k padded with 0)"""
    scale = n_in / n_out
    fs = max(scale, 1.0)
    support = SUPPORT[flt] * fs
    xmins, ns, ks = [], [], []
    for o in range(n_out):
        center = (o + 0.5) * scale
        ss = 1.0 / fs
        xmin = max(int(center - support + 0.5), 0)
        n = min(int(center + support + 0.5), n_in) - xmin
        w = [_filter(flt, (x + xmin - center + 0.5) * ss) for x in range(n)]
        ww = 0.0
        for v in w:
            ww += v
        if ww != 0.0:
            w = [v / ww for v in w]
        ks.append([int(-0.5 + v * (1 << PRECISION_BITS)) if v < 0 else int(0.5 + v * (1 << PRECISION_BITS)) for v in w])
        xmins.append(xmin)
        ns.append(n)
    k = np.zeros((n_out, max(ns)), np.int64)
    for o, row in enumerate(ks):
        k[o, : len(row)] = row
    return np.array(xmins, np.int64), np.array(ns, np.int64), k


def _pass(a: np.ndarray, n_out: int, flt: int) -> np.ndarray:
    """one pass along the last axis of an int64 array of 8-bit values, clipped to 8 bits"""
    xmin, n, k = coeffs(a.shape[-1], n_out, flt)
    # every partial sum of Pillow's 32-bit accumulator is bounded by 2^21 + 255 * sum |k|
    assert (1 << 21) + 255 * int(np.abs(k).sum(axis=1).max()) < 1 << 31
    s = np.full(a.shape[:-1] + (n_out,), 1 << (PRECISION_BITS - 1), np.int64)
    for t in range(k.shape[1]):
        idx = np.minimum(xmin + t, a.shape[-1] - 1)
        s += a[..., idx] * np.where(t < n, k[:, t], 0)
    return np.clip(s >> PRECISION_BITS, 0, 255)


def resize_plane(p: np.ndarray, w_out: int, h_out: int, flt: int) -> np.ndarray:
    """Image.fromarray(p, "L").resize((w_out, h_out), flt): horizontal pass first, no pass on an axis that keeps its size"""
    assert p.ndim == 2 and flt in FILTERS
    t = p.astype(np.int64)
    if w_out != p.shape[1]:
        t = _pass(t, w_out, flt)
    if h_out != p.shape[0]:
        t = _pass(t.T, h_out, flt).T
    return np.ascontiguousarray(t.astype(np.uint8))


def resize_planar(y, u, v, w_out: int, h_out: int, fmt: int, flt: int):
    """R(frame) of a planar frame: (y, u, v) of the w_out x h_out frame at chroma format fmt"""
    from h2j_b200 import chroma_shape

    ch, cw = chroma_shape(w_out, h_out, fmt)
    return resize_plane(y, w_out, h_out, flt), resize_plane(u, cw, ch, flt), resize_plane(v, cw, ch, flt)


def resize_semiplanar(y, uv, w_out: int, h_out: int, fmt: int, flt: int):
    """R(frame) of a semi-planar frame (uv: rows of interleaved Cb/Cr pairs): the resized PLANAR frame"""
    assert uv.ndim == 2 and uv.shape[1] % 2 == 0
    return resize_planar(y, uv[:, 0::2], uv[:, 1::2], w_out, h_out, fmt, flt)
