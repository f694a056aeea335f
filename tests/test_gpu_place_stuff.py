"""GPU suite: scan placement (K4b, scan_place_kernel) and byte stuffing (K5, stuff_kernel) at their word, unit, group and
chunk boundaries.  Every case of tests/support/scan_model.py -- each holds the edge it is named after, which
tests/test_place_stuff_cases.py asserts -- is encoded and must give the oracle's JPEG byte for byte, its scan_bits,
stuffed_ff and header_bytes, and entropy-decode to the oracle's coefficients.

K4b has two forms: a warp concatenates 8 units when a launch has fewer groups than two per SM, 32 otherwise.  Every case
runs in both, alone in its batch (the 8 form) and repeated until the batch's groups reach twice the SM count (the 32
form), as one batch of every K4b case at once (frames of different group counts in one launch), and in part at 4:2:2 and
4:4:4.  The comment sweep moves the scan through all 16 offsets of K5's output line; the longest comment fills the COM
segment's length field."""
import numpy as np
import pytest

from tests.support import scan_model as M
from tests.support.layouts import Frames, desc, planar

pytestmark = pytest.mark.gpu

FORMS = (8, 32)


def _sm_count():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


def _batch(groups, form):
    """frames of `groups` K4b groups each for a launch in the given form"""
    limit = 2 * _sm_count()
    n = 1 if form == 8 else -(-limit // groups)
    assert (groups * n < limit) == (form == 8), (groups, n, limit)
    return n


def _frame(case):
    return np.concatenate([p.reshape(-1) for p in case.planes])


def _cap(jpegs):
    return max(len(j) for j in jpegs) + 65536


def _check(orc, e, res, cases):
    """the batch's JPEGs and frame records against the oracle's, frame by frame"""
    assert res.status == [0] * len(cases)
    for i, c in enumerate(cases):
        s = c.scan
        assert res.jpegs[i] == s.jpeg, f"{c.name} (chroma format {c.chroma_format}), frame {i} of {len(cases)}"
        fi = e.frame_info(0, i)
        assert (fi.scan_bits, fi.stuffed_ff, fi.header_bytes) == (s.scan_bits, s.stuffed_ff, s.header_bytes), (c.name, i)
    first = {}
    for i, c in enumerate(cases):
        first.setdefault(id(c), i)
    for i in first.values():
        levels, _ = orc.decode_coefs(res.jpegs[i])
        assert (levels == cases[i].scan.coefs).all(), cases[i].name


def _encode_repeated(orc, case, form):
    import torch

    import h2j_b200

    w, h = case.size
    n = _batch(case.scan.groups, form)
    frame = _frame(case)
    d = torch.from_numpy(frame).cuda().repeat(n)
    with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=n, n_slots=1, fixed_qscale=case.qscale, chroma_format=case.chroma_format,
                          max_jpeg_bytes=_cap([case.scan.jpeg]), comment=case.comment) as e:
        e.submit_device(0, d.data_ptr(), frame.size, n, w, h)
        _check(orc, e, e.collect(0), [case] * n)


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("name", list(M.EDGES))
def test_edge_case(orc, name, form):
    _encode_repeated(orc, M.case(name), form)


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("name", M.FORMAT_EDGES)
@pytest.mark.parametrize("chroma_format", [1, 2])
def test_edge_case_other_formats(orc, chroma_format, name, form):
    _encode_repeated(orc, M.case(name, chroma_format), form)


@pytest.mark.parametrize("form", FORMS)
def test_k4b_cases_in_one_list_batch(orc, form):
    """every K4b case in one h2j_submit_device_list batch: groups_per_frame is the largest frame's, the other frames' tickets
    past their own groups return at once"""
    import h2j_b200 as h2j

    base = [M.case(k) for k in M.K4B_EDGES + M.SIZE_EDGES]
    groups = max(c.scan.groups for c in base)
    assert len({c.scan.groups for c in base}) >= 3
    reps = -(-_batch(groups, form) // len(base)) if form == 32 else 1
    cases = base * reps
    assert (groups * len(cases) < 2 * _sm_count()) == (form == 8)
    fr = Frames()
    descs = [desc(fr, y, u, v, *planar(y, u)) for y, u, v in (c.planes for c in cases)]
    w, h = max(c.size[0] for c in base), max(c.size[1] for c in base)
    with h2j.Encoder(max_width=w, max_height=h, max_batch=len(cases), n_slots=1, fixed_qscale=M.QSCALE,
                     max_jpeg_bytes=_cap([c.scan.jpeg for c in base])) as e:
        e.submit_device_list(0, h2j.LAYOUT_PLANAR, descs)
        _check(orc, e, e.collect(0), cases)


@pytest.mark.parametrize("length", range(16))
def test_comment_sweep_moves_every_line_offset(orc, length):
    """header_bytes + 0xFF bytes in front of a chunk, mod 16, is where K5's image of the chunk starts in its output line"""
    _encode_repeated(orc, M.comment_case(length), 8)


def test_longest_comment(orc):
    import h2j_b200

    y, u, v = M.textured(0, 320, 240, 5)
    text = bytes(b"abcdefghijklmnopqrstuvwxyz"[i % 26] for i in range(M.MAX_COMMENT))
    want, dbg, coefs = orc.oracle_encode(y, u, v, comment=text, want_coefs=True)
    assert want[4:6] == b"\xff\xff"
    with h2j_b200.Encoder(max_width=320, max_height=240, max_batch=1, n_slots=1, comment=text) as e:
        frame = orc.pack_i420(y, u, v)[None, :].copy()
        e.submit_host(0, frame.ctypes.data, frame.shape[1], 1, 320, 240)
        res = e.collect(0)
        got = res.jpegs[0]
        fi = e.frame_info(0, 0)
    assert got == want
    assert (fi.header_bytes, fi.scan_bits) == (dbg.header_bytes, dbg.scan_bits)
    assert (orc.decode_coefs(got)[0] == coefs).all()
