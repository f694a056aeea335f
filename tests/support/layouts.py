"""Device frames for the GPU tests: planes placed into a padded buffer at any layout a caller or a hardware decoder uses,
uploaded as one batch or as frames in their own allocations, and the encoder calls the tests make on them.

Pitches and offsets are in bytes.  Padding is PAD: a padding byte that reached a picture would change its JPEG.
TEST INFRASTRUCTURE ONLY."""
import numpy as np
from numpy.lib.stride_tricks import as_strided

PAD = 0xA5
GUARD = 64
BIG_JPEG = 8 * 1024 * 1024

# (w, h, kind, amp): partial MCUs, partial tiles, 2x2 .. 1080p
CASES = [(16, 16, "textured", 40), (2, 2, "noise", 100), (17, 17, "noise", 60), (33, 47, "blocks", 30), (64, 64, "binary", 0), (131, 77, "textured", 80),
         (322, 242, "textured", 40), (641, 479, "noise", 20), (8, 16, "noise", 50), (9, 31, "noise", 50), (1280, 720, "textured", 30),
         (1918, 1078, "textured", 40), (1920, 1080, "ff", 0)]


def align(x, a):
    return (x + a - 1) // a * a


def place(y, u, v, y_pitch, c_pitch, u_off, v_off=None, size=None, pad=PAD):
    """Planes (uint8 or uint16) -> the frame's bytes (uint8): luma rows y_pitch apart from 0, then Cb rows at u_off and Cr
    rows at v_off, c_pitch apart; v_off None: semi-planar, rows of Cb/Cr pairs at u_off.  The buffer holds `size` bytes;
    size None: it ends at the last sample of the plane that reaches furthest."""
    if v_off is None:
        uv = np.empty((u.shape[0], 2 * u.shape[1]), u.dtype)
        uv[:, 0::2], uv[:, 1::2] = u, v
        planes = [(0, y_pitch, y), (u_off, c_pitch, uv)]
    else:
        planes = [(0, y_pitch, y), (u_off, c_pitch, u), (v_off, c_pitch, v)]
    rows = [(off, pitch, np.ascontiguousarray(p).view(np.uint8)) for off, pitch, p in planes]
    end = max(off + pitch * (b.shape[0] - 1) + b.shape[1] for off, pitch, b in rows)
    buf = np.full(end if size is None else size, pad, np.uint8)
    assert end <= buf.size, (end, buf.size)
    for off, pitch, b in rows:
        as_strided(buf[off:], shape=b.shape, strides=(pitch, 1))[:] = b
    return buf


def planar(y, u, y_pitch=None, c_pitch=None, gap=0):
    """(y_pitch, c_pitch, u_off, v_off) of a planar frame whose planes lie one behind the other, each followed by `gap`
    spare rows (a decoder surface taller than the picture); pitches default to the rows' lengths"""
    (h, w), (ch, cw) = y.shape, u.shape
    y_pitch, c_pitch = y_pitch or w * y.itemsize, c_pitch or cw * u.itemsize
    u_off = y_pitch * (h + gap)
    return y_pitch, c_pitch, u_off, u_off + c_pitch * (ch + gap)


def semiplanar(y, pitch, gap=0):
    """(y_pitch, c_pitch, uv_off) of a semi-planar frame at one pitch, the pair plane behind the luma rows and `gap` spare rows"""
    return pitch, pitch, pitch * (y.shape[0] + gap)


def upload(frames, stride, shift=0):
    """frames (1-D uint8 arrays, each at most `stride` long) -> one device allocation, frame i at byte shift + i * stride and
    PAD between.  Returns (tensor that owns the memory, device address of frame 0)."""
    import torch

    host = np.full(shift + len(frames) * stride, PAD, np.uint8)
    for i, f in enumerate(frames):
        host[shift + i * stride: shift + i * stride + len(f)] = f
    d = torch.from_numpy(host).cuda()
    torch.cuda.synchronize()  # the slot runs on its own stream
    return d, d.data_ptr() + shift


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


def desc(fr, y, u, v, y_pitch, c_pitch, u_off, v_off=None, size=None, shift=0):
    """the h2j_b200.FrameDesc of place(y, u, v, y_pitch, c_pitch, u_off, v_off, size), put into its own allocation by `fr`"""
    import h2j_b200

    h, w = y.shape
    data = fr.put(place(y, u, v, y_pitch, c_pitch, u_off, v_off, size), shift)
    return h2j_b200.FrameDesc(data, w, h, y_pitch, c_pitch, u_off, 0 if v_off is None else v_off)


def encoder(fmt, max_batch, **kw):
    """an encoder of one slot, 1920 x 1088 and JPEGs of up to BIG_JPEG bytes unless kw says otherwise"""
    import h2j_b200

    kw.setdefault("max_jpeg_bytes", BIG_JPEG)
    return h2j_b200.Encoder(max_width=kw.pop("max_width", 1920), max_height=kw.pop("max_height", 1088), max_batch=max_batch, n_slots=1,
                            chroma_format=fmt, **kw)


def run(e, submit, n):
    """submit, collect; returns (jpegs, kernel launches the batch took)"""
    before = e.kernel_launches
    submit()
    res = e.collect(0)
    assert res.status == [0] * n
    return res.jpegs, e.kernel_launches - before


def pipeline_launches(e):
    """launches of a planar submit that needs no copy: the pipeline plus the pack at collect"""
    import torch

    import h2j_b200

    w = h = 16
    ch, cw = h2j_b200.chroma_shape(w, h, e.chroma_format)
    d = torch.zeros(align(w * h + 2 * cw * ch, 256), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    before = e.kernel_launches
    e.submit_device(0, d.data_ptr(), d.numel(), 1, w, h)
    assert e.collect(0).status == [0]
    return e.kernel_launches - before
