"""CPU suite: the frame layouts the GPU tests place their planes at (tests/support/layouts.py), on buffers written out by
hand."""
import numpy as np

from tests.support.layouts import PAD, place, planar, semiplanar

P = PAD


def test_nv12_at_a_pitch():
    y = np.array([[1, 2, 3], [4, 5, 6]], np.uint8)
    u, v = np.array([[7, 8]], np.uint8), np.array([[9, 10]], np.uint8)
    assert semiplanar(y, 8) == (8, 8, 16)
    assert place(y, u, v, 8, 8, 16, size=24).tolist() == [1, 2, 3, P, P, P, P, P,
                                                           4, 5, 6, P, P, P, P, P,
                                                           7, 9, 8, 10, P, P, P, P]
    # without a size the buffer ends at the last sample; behind a spare luma row
    assert place(y, u, v, *semiplanar(y, 4, gap=1)).tolist() == [1, 2, 3, P, 4, 5, 6, P, P, P, P, P, 7, 9, 8, 10]


def test_planar_16_bit_cr_in_front_of_cb():
    y = np.array([[0x0102, 0x0304], [0x0506, 0x0708]], np.uint16)
    u, v = np.array([[0x090A]], np.uint16), np.array([[0x0B0C]], np.uint16)
    assert place(y, u, v, 6, 4, 16, 12).tolist() == [2, 1, 4, 3, P, P,
                                                     6, 5, 8, 7, P, P,
                                                     0xC, 0xB, P, P,
                                                     0xA, 9]
    assert place(y, u, v, *planar(y, u), pad=0).tolist() == [2, 1, 4, 3, 6, 5, 8, 7, 0xA, 9, 0xC, 0xB]
