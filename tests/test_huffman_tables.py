"""CPU suite: the oracle's Huffman table builder (orc_huffman_table, libavcodec's mjpegenc_huffman.c restated) on
adversarial histograms, against properties that do not depend on tie order, computed with exact Python integers --
among them the optimal cost of a 16-bit length-limited prefix code from a textbook package-merge."""
import numpy as np
import pytest

from tests.support import histograms as H


@pytest.fixture(scope="module")
def tables():
    dc, ac = H.generate()
    return dc + ac


def test_generator_covers_its_families(tables):
    kinds = {k for k, _ in tables}
    for k in ("few1", "few2", "few3", "equal", "equal_all_k", "two_valued", "duplicated", "ascending", "descending",
              "fibonacci", "pow2", "ac_zipf", "all256_random", "all256_equal"):
        assert k in kinds, k
    used = [int((h != 0).sum()) for _, h in tables]
    assert min(used) == 1 and max(used) == 256
    assert set(range(2, 257)) <= {int((h != 0).sum()) for k, h in tables if k == "equal_all_k"}
    assert max(int(h.astype(np.int64).sum()) for _, h in tables) >= 10 ** 8
    assert len(tables) == 2000
    # exact ties between a symbol's count and a package sum at some level: there the tie rule decides the lengths
    assert sum(H.symbol_package_ties(h[h != 0]) > 0 for _, h in tables) >= 200
    # the same seed gives the same histograms
    again = H.generate()
    assert all((a[1] == b[1]).all() for a, b in zip(tables, again[0] + again[1]))


def test_reference_optimum_on_small_cases():
    # unlimited Huffman on (1, 1, 2) plus the zero leaf: lengths 3, 3, 2, 1 -> 0*3 + 1*3 + 1*2 + 2*1 ... = 7
    assert H.optimal_cost([1, 1, 2]) == 7
    # one symbol: it and the zero leaf get one bit each
    assert H.optimal_cost([5]) == 5
    # 17 equal counts need 5 bits for some; the limit does not bind
    assert H.optimal_cost([1] * 17, max_len=16) == H.optimal_cost([1] * 17, max_len=40)
    # Fibonacci counts: unlimited depth is ~n, the 16-bit limit must cost more than the unlimited optimum
    f = [1, 1]
    while len(f) < 30:
        f.append(f[-1] + f[-2])
    assert H.optimal_cost(f, max_len=16) > H.optimal_cost(f, max_len=64)
    # brute force over every length assignment of 4 symbols + the zero leaf with Kraft <= 1, limit 3
    import itertools
    counts = [3, 5, 7, 11]
    best = min(sum(c * l for c, l in zip(counts + [0], ls)) for ls in itertools.product(range(1, 4), repeat=5)
               if sum(2.0 ** -l for l in ls) <= 1)
    assert H.optimal_cost(counts, max_len=3) == best


def test_oracle_tables_are_optimal_length_limited_codes(orc, tables):
    deep = 0
    for i, (kind, hist) in enumerate(tables):
        bits, vals, nv = H.oracle_table(orc, hist)
        bad = H.check_table(hist, bits, vals, nv)
        assert not bad, (i, kind, bad)
        deep += int(bits[16]) > 0
    assert deep >= 50, "the histograms should force many tables to the 16-bit limit"


def test_length_limit_cuts_many_levels(orc):
    """43 Fibonacci counts: an unlimited Huffman code would be 43 deep; at 16 bits the limit decides most lengths."""
    f = [1, 1]
    while len(f) < 43:
        f.append(f[-1] + f[-2])
    hist = np.zeros(256, np.uint32)
    hist[:43] = f
    bits, vals, nv = H.oracle_table(orc, hist)
    assert not H.check_table(hist, bits, vals, nv)
    assert int(bits[16]) >= 15 and sum(int(b) for b in bits[1:17]) == 43
