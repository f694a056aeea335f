"""GPU suite: the host batch scope (host/Encoder.cpp) with pictures of several sizes interleaved.  A job holds pictures of
any sizes, so the scope hands over full batches instead of sealing one on every size change; every file is byte-identical
to the oracle's JPEG."""
import ctypes as C
import os

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST_SO = os.path.join(ROOT, "h264-h265-to-jpeg_b200", "lib", "libh2j_host.so")


def test_interleaved_sizes_share_batches(orc, tmp_path):
    lib = C.CDLL(HOST_SO)
    lib.h2j_host_yuv2jpeg_file.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_char_p]
    lib.h2j_host_batch_end.argtypes = [C.POINTER(C.c_int)]
    sizes = [(322, 242), (1280, 720), (641, 479)] * 7  # 21 pictures, three sizes interleaved, the smallest first
    assert lib.h2j_host_batch_begin(8) == 0
    want, outs = [], []
    for i, (w, h) in enumerate(sizes):
        y, u, v = orc.synth_planes(w, h, "textured", seed=300 + i, amp=20 + i)
        out = str(tmp_path / f"m_{i}.jpeg")
        assert lib.h2j_host_yuv2jpeg_file(y.ctypes.data, y.strides[0], u.ctypes.data, u.strides[0], v.ctypes.data, v.strides[0], w, h, 0,
                                          out.encode()) == 1
        want.append(orc.oracle_encode(y, u, v)[0])
        outs.append(out)
    failed = C.c_int(-1)
    assert lib.h2j_host_batch_end(C.byref(failed)) == len(sizes) and failed.value == 0
    assert lib.h2j_host_batches_submitted() == (len(sizes) + 7) // 8
    for out, w_ in zip(outs, want):
        assert open(out, "rb").read() == w_
