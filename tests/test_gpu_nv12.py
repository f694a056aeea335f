"""GPU suite: NV12 device input (DESIGN.md row (f)(2)).  The reference has no NV12 input -- its decoder is libavcodec's
software decoder and hands over yuv420p -- so parity is defined through the equivalent planar frame: the JPEG of an NV12
frame must be byte-identical to the oracle's JPEG of the yuv420p frame with the same samples."""
import pytest

from tests.support.layouts import place, upload

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize(
    "w,h,pitch_align,extra_rows,kind",
    [
        (1920, 1080, 256, 8, "textured"),   # NVDEC-like: pitch 2048, chroma plane behind 1088 luma rows
        (1918, 1078, 1, 0, "textured"),     # tight, nothing aligned: the byte paths
        (322, 242, 16, 0, "noise"),
        (17, 9, 1, 0, "noise"),             # odd width and height: ceil(w/2) pairs, ceil(h/2) chroma rows
        (64, 48, 64, 3, "const"),
        (330, 241, 8, 1, "noise"),          # read in place: right edge cuts an MCU's pairs, odd height (ch = h >> 1 rows are read)
        (1280, 720, 128, 0, "textured"),    # read in place, tiles wrap MCU rows
        (48, 16, 8, 0, "noise"),            # a single MCU row, three MCUs: less than one tile
    ],
)
def test_nv12_matches_planar(orc, w, h, pitch_align, extra_rows, kind):
    import torch

    import h2j_b200

    n = 3
    cw = (w + 1) // 2
    row = max(w, 2 * cw)
    pitch = (row + pitch_align - 1) // pitch_align * pitch_align
    uv_off = pitch * (h + extra_rows)
    frames, want = [], []
    for s in range(n):
        y, u, v = orc.synth_planes(w, h, kind, seed=40 + s)
        frames.append(place(y, u, v, pitch, pitch, uv_off, size=uv_off + pitch * u.shape[0]))
        want.append(orc.oracle_encode(y, u, v)[0])
    stride = (len(frames[0]) + 255) // 256 * 256
    d, ptr = upload(frames, stride)
    with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=n, n_slots=1) as e:
        e.submit_device_nv12(0, ptr, stride, pitch, uv_off, n, w, h)
        res = e.collect(0)
        assert res.status == [0] * n
        for i in range(n):
            assert res.jpegs[i] == want[i], f"frame {i}: NV12 JPEG differs from the oracle's JPEG of the planar frame"
        # an unaligned base address takes the byte path and must give the same bytes
        d2 = torch.zeros(n * stride + 1, dtype=torch.uint8, device="cuda")
        d2[1:] = d.reshape(-1)
        # d2 is produced on torch's current stream, the slot runs on its own: order the slot behind the producer
        # (include/h2j_b200.h, "Stream ordering of device inputs")
        ev = torch.cuda.Event()
        ev.record()
        e.wait_event(0, ev.cuda_event)
        e.submit_device_nv12(0, d2.data_ptr() + 1, stride, pitch, uv_off, n, w, h)
        res2 = e.collect(0)
        assert res2.jpegs == res.jpegs


def test_nv12_in_place_with_range_conversion_and_fixed_qscale(orc):
    """The in-place path through the limited->full LUT (bytewise predecessor rows, LUT on traded samples) and at a fixed
    quantiser."""
    import h2j_b200

    w, h, pitch = 322, 242, 384
    y, u, v = orc.synth_planes(w, h, "textured", seed=77)
    fr = place(y, u, v, pitch, pitch, pitch * h, size=pitch * (h + u.shape[0]))
    d, ptr = upload([fr], len(fr))
    for kw, okw in (({"range_mode": 1}, {"range_mode": 1}), ({"fixed_qscale": 3}, {"fixed_qscale": 3})):
        with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=1, n_slots=1, **kw) as e:
            e.submit_device_nv12(0, ptr, len(fr), pitch, pitch * h, 1, w, h)
            got = e.collect(0).jpegs[0]
        assert got == orc.oracle_encode(y, u, v, **okw)[0], kw
