"""CPU: the dispatch matrix (tests/support/dispatch.py) runs every kernel the library compiles, holds every valid pair of
its parameters and the required launch shapes, and its model follows the launch-shape rules of h2j_api.cu."""
import itertools
import re

import pytest

from tests.support import dispatch as D

@pytest.fixture(scope="module")
def cases():
    return D.matrix()


def test_the_matrix_runs_every_compiled_kernel(cases):
    want = D.compiled_kernels()
    got = set().union(*(D.model(c)["kernels"] for c in cases))
    assert len(want) >= 51
    assert not want - got, f"compiled kernels no case of the matrix runs: {sorted(want - got)}"
    assert not got - want, f"kernels the model names that the library does not compile: {sorted(got - want)}"


def test_every_valid_pair_is_covered(cases):
    space = [p for p in itertools.product(D.FMTS, [p.name for p in D.PATHS], D.FORMS, D.TILES, D.K4B, D.SETTINGS)
             if D.valid(p[0], D.BY_NAME[p[1]], *p[2:])]
    want = set().union(*(D.pairs(p) for p in space))
    got = set().union(*(D.pairs(c.params()) for c in cases if c.path.name in D.BY_NAME))
    missing = sorted(want - got)
    assert not missing, f"{len(missing)} pairs uncovered, e.g. {missing[:5]}"
    # every value of every parameter occurs, and the cases hold the K4b form and batch form they name
    for c in cases:
        m = D.model(c)
        assert m["k4b"] in (None, c.k4b) and m["list"] == (c.form == "list"), c.id
    assert 150 <= len(cases) <= 260, len(cases)


def k2_name(fmt, nv12, lst):
    b = D.bool_name
    return f"h2j::fdct_quant_kernel<{b(nv12)}, {b(lst)}>" if fmt == 0 else f"h2j::fdct_quant_fmt_kernel<{fmt}, {b(nv12)}, {b(lst)}>"


def test_every_fdct_instantiation_walks_several_tiles_with_a_partial_last_group(cases):
    want = {k for k in D.compiled_kernels() if "fdct_quant" in k}
    got = set()
    for c in cases:
        m = D.model(c)
        if m["tiles_per_cta"] and m["tiles_per_cta"] > 1 and D.partial_last_group(c):
            got |= {k for k in m["kernels"] if "fdct_quant" in k}
    assert not want - got, f"FDCT kernels never run with several tiles per CTA on a partial last group: {sorted(want - got)}"


def test_every_input_kernel_runs_in_the_list_form_on_two_sizes(cases):
    # depth_to_8_kernel has no list call: 16-bit frames come in one layout at one stride
    want = {k for k in D.compiled_kernels() if re.match(r"h2j::(repitch|nv12_to_i420|downscale_list|rgb_to_planar|resize_list)_kernel", k)}
    got = {D.model(c)["copy"] for c in cases if D.model(c)["list"] and len(set(c.out_sizes())) >= 2}
    assert not want - got, f"input kernels never run in the list form: {sorted(want - got)}"


def test_the_production_and_fallback_paths_are_in_the_matrix(cases):
    # semi-planar decoder surfaces listed and read in place with the automatic tiles per CTA above 1, every chroma format
    for fmt in D.FMTS:
        assert any(c.fmt == fmt and c.path.kind == "sp" and c.tiles == 0 and D.model(c)["list"] and D.model(c)["copy"] is None
                   and D.model(c)["tiles_per_cta"] > 1 for c in cases), fmt
    # unaligned planar frames read in place, device and host, in both forms and every chroma format
    in_place = [c for c in cases if dict(c.path.knob).get("planar_copy") == 0 and not all(D.frame_aligned8(c, f) for f in c.frames)]
    assert {(c.fmt, c.path.kind, c.form) for c in in_place} >= {(f, "planar", form) for f in D.FMTS for form in D.FORMS}
    assert {c.fmt for c in in_place if c.path.kind == "host"} == set(D.FMTS)


# tiles per CTA: total tiles x roles // (SMs x 16 x 4), clamped to 1 .. 16 (h2j_api.cu launch_pipeline)
@pytest.mark.parametrize("sizes,fmt,sms,want", [
    ([(1920, 1080)] * 7, 0, 148, 1),      # 7 x 510 tiles x 3 roles = 10,710 < 2 x 9,472
    ([(1920, 1080)] * 13, 0, 148, 2),     # 19,890
    ([(3840, 2160)] * 13, 0, 148, 8),     # 13 x 2,025 x 3 = 78,975
    ([(1920, 1080)] * 64, 1, 148, 13),    # 64 x 510 x 4 = 130,560
    ([(1920, 1080)] * 256, 0, 148, 16),   # 391,680: clamped
    ([(2, 2)], 2, 148, 1),
    ([(1920, 1080)] * 13, 2, 148, 4),     # 13 x 1,020 x 3 = 39,780
    ([(1920, 1080)] * 13, 0, 132, 2),     # 19,890 // 8,448
])
def test_tiles_per_cta_rule(sizes, fmt, sms, want):
    assert D.tiles_per_cta(sizes, fmt, sms) == want
    assert D.tiles_per_cta(sizes, fmt, sms, forced=3) == 3


# K4b: 8 units per warp while groups of 256 units per frame (of the largest frame) x frames < 2 x SMs
@pytest.mark.parametrize("sizes,fmt,sms,want", [
    ([(1920, 1080)] * 49, 0, 148, 8),     # 1,530 units: 6 groups; 294 < 296
    ([(1920, 1080)] * 50, 0, 148, 32),    # 300
    ([(3840, 2160)] * 12, 0, 148, 8),     # 6,075 units: 24 groups; 288
    ([(3840, 2160)] + [(2, 2)] * 12, 0, 148, 32),  # 312: the largest frame counts for every frame
    ([(3840, 2160)] * 6, 2, 148, 8),      # 4:4:4: 12,150 units, 48 groups; 288
    ([(3840, 2160)] * 7, 2, 148, 32),     # 336
    ([(64, 64), (131, 77)], 0, 148, 8),
    ([(1920, 1080)] * 64, 1, 148, 32),    # 2,040 units: 8 groups; 512
])
def test_k4b_width_rule(sizes, fmt, sms, want):
    assert D.k4b_width(sizes, fmt, sms) == want
