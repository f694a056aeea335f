"""CPU suite: the frames of tests/test_gpu_place_stuff.py hold the boundaries of scan placement (K4b) and byte stuffing (K5)
they are meant to, by the oracle alone (tests/support/scan_model.py), so that none of them can silently stop exercising
its edge; and the model they are described with agrees with the oracle's JPEGs."""
import numpy as np
import pytest

from tests.support import scan_model as M


@pytest.mark.parametrize("name", list(M.EDGES))
def test_case_has_its_edge(name):
    c = M.case(name)
    assert M.EDGES[name](c.scan), name


@pytest.mark.parametrize("name", M.FORMAT_EDGES)
@pytest.mark.parametrize("chroma_format", [1, 2])
def test_case_has_its_edge_in_other_formats(name, chroma_format):
    c = M.case(name, chroma_format)
    assert M.EDGES[name](c.scan), (name, chroma_format)


def test_the_k4b_forms_see_their_boundaries():
    """group firsts with c == 0 and with a carry over two staged words; run firsts inside a group with and without one"""
    s = M.case("group_first_hiw").scan
    assert s.groups >= 2
    firsts = np.arange(M.GROUP_UNITS, s.n_units, M.GROUP_UNITS)
    u = firsts[s.hiw[firsts]][0]
    assert s.carry[u] > s.last_word_bits[u - 1] and s.unit_bits[u - 1] % 32 != 0
    assert (M.case("group_first_c0").scan.group_start[1:] % 32 == 0).any()
    w = M.case("unit_words").scan.words
    assert {32, 63, 64} <= set(w.tolist()) and w.max() > 96


def test_unit_counts_around_group_boundaries():
    for n, groups, last in ((255, 1, 255), (256, 1, 256), (257, 2, 1), (512, 2, 256), (513, 3, 1)):
        s = M.case(f"units_{n}").scan
        assert (s.n_units, s.groups, s.n_units - M.GROUP_UNITS * (s.groups - 1)) == (n, groups, last)


def test_frame_ends():
    assert M.case("end_word_aligned").scan.scan_bits % 32 == 0
    s = M.case("padding_makes_ff").scan
    pad = 8 - s.scan_bits % 8
    assert s.data[-1] & ((1 << pad) - 1) == (1 << pad) - 1  # the padding is ones ...
    assert s.jpeg.endswith(b"\xff\x00\xff\xd9")              # ... and the 0xFF it completes is stuffed before EOI
    assert {M.case(f"bytes_mod16_{r}").scan.n_bytes % 16 for r in range(16)} == set(range(16))
    for n, chunks in ((4096, 1), (4097, 2), (8192, 2), (8193, 3)):
        s = M.case(f"bytes_{n}").scan
        assert (s.n_bytes, s.n_chunks) == (n, chunks)


def test_k5_chunks():
    assert [M.case(f"chunks_{k}").scan.n_chunks for k in ("1", "32")] == [1, 32]
    assert M.case("chunks_over_64").scan.n_chunks > 2 * 32
    s = M.case("ff_at_chunk_ends").scan
    k = np.arange(1, s.n_chunks) * M.CHUNK_BYTES
    assert (s.data[k - 1] == 0xFF).any() and (s.data[k] == 0xFF).any()


def test_every_line_offset_under_the_comment_sweep():
    """header_bytes grows by one per comment character, so chunk 0 starts at all 16 offsets of its output line"""
    cases = [M.comment_case(n) for n in range(16)]
    hb = [c.scan.header_bytes for c in cases]
    assert hb == list(range(hb[0], hb[0] + 16))
    assert {int(c.scan.a0[0]) for c in cases} == set(range(16))
    assert all((c.scan.data == cases[0].scan.data).all() for c in cases)  # the scan is the same


def test_model_matches_the_oracle_jpeg():
    """the model's stuffed-byte count and chunk census against the JPEG itself"""
    for name in ("ff_at_chunk_ends", "zero_chunk_before_counts", "bytes_4097"):
        s = M.case(name).scan
        assert len(s.jpeg) == s.header_bytes + s.n_bytes + s.stuffed_ff + 2
        assert s.chunk_ff.sum() == s.stuffed_ff == s.jpeg[s.header_bytes:].count(b"\xff\x00")
        assert s.a0[-1] == (s.header_bytes + s.stuffed_ff - s.chunk_ff[-1]) % 16


def test_longest_comment_fits_its_length_field(orc):
    y = np.full((16, 16), 128, np.uint8)
    u = np.full((8, 8), 128, np.uint8)
    jpeg, dbg, _ = orc.oracle_encode(y, u, u, comment=b"c" * M.MAX_COMMENT)
    assert jpeg[2:6] == b"\xff\xfe\xff\xff" and dbg.header_bytes > M.MAX_COMMENT
