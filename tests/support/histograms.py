"""Seeded symbol histograms for the Huffman table builders, and the plain references they are checked with.

The histograms sit where the table construction is at its limits: one to three symbols, many equal counts (the tie
order of both sorts alone decides HUFFVAL), sorted input, Fibonacci and power-of-two counts (deep length-limit cuts and
exact ties between a symbol and a package sum), Zipf-like AC tables, all 256 byte values, totals up to ~10^8.
TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import numpy as np

MAX_LEN = 16
# the symbols a real AC table can hold: EOB, ZRL and (run, size) for run 0..15, size 1..10
AC_SYMBOLS = np.array([0x00, 0xF0] + [(r << 4) | s for r in range(16) for s in range(1, 11)], np.int64)
DC_SYMBOLS = np.arange(16)  # a DC code table has 16 entries (the encoder uses sizes 0..11)


def package_sums_max(counts) -> int:
    """Largest item weight of the 16 package-merge levels libavcodec runs over counts + one zero-count leaf."""
    leaves = sorted([int(c) for c in counts] + [0])
    prev, top = leaves, max(leaves)
    for t in range(1, MAX_LEN + 1):
        pk = [prev[2 * i] + prev[2 * i + 1] for i in range(len(prev) // 2)]
        prev = sorted((leaves if t < MAX_LEN else []) + pk)
        top = max([top] + pk)
    return top


def symbol_package_ties(counts) -> int:
    """How often, over the levels that take symbols, a symbol's count equals a package sum of the same level."""
    leaves = sorted([int(c) for c in counts] + [0])
    prev, ties = leaves, 0
    for _ in range(1, MAX_LEN):
        pk = [prev[2 * i] + prev[2 * i + 1] for i in range(len(prev) // 2)]
        ties += len(set(leaves) & set(pk))
        prev = sorted(leaves + pk)
    return ties


def _fib(n):
    a, b, out = 1, 1, []
    for _ in range(n):
        out.append(a)
        a, b = b, a + b
    return out


class _Gen:
    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.out = []  # (kind, hist[256] uint32)

    def add(self, kind, syms, counts):
        syms = np.asarray(syms, np.int64)
        counts = np.asarray(counts, np.int64)
        assert len(syms) == len(counts) and len(np.unique(syms)) == len(syms) and (counts > 0).all(), kind
        assert package_sums_max(counts) < 2 ** 31, kind  # libavcodec's int fields are defined there
        h = np.zeros(256, np.uint32)
        h[syms] = counts
        self.out.append((kind, h))

    def syms(self, pool, k):
        return self.rng.choice(pool, size=k, replace=False)

    def scale(self, counts, total):
        c = np.asarray(counts, np.float64)
        return np.maximum(1, np.round(c * (total / c.sum()))).astype(np.int64)


def _families(g: _Gen, pool, kmax, reps):
    r = g.rng
    big = [1, 2, 7, 1000, 10 ** 6, 5 * 10 ** 7]

    def top(k):  # a large count, but k of them stay far below 2^31
        return int(min(r.choice(big), 2 ** 28 // k))

    for _ in range(reps):
        for k in (1, 2, 3):  # zero used symbols cannot occur: every block codes a DC size and ends in EOB or level 63
            g.add(f"few{k}", g.syms(pool, k), r.integers(1, top(k) + 1, k))
        k = int(r.integers(2, kmax + 1))  # all counts equal: only the sorts' tie order decides HUFFVAL
        g.add("equal", g.syms(pool, k), np.full(k, top(k)))
        k = int(r.integers(2, kmax + 1))
        a, b = sorted(int(x) for x in r.integers(1, 10 ** int(r.integers(1, 7)), 2))
        g.add("two_valued", g.syms(pool, k), r.choice([a, b + 1], k))
        k = int(r.integers(4, kmax + 1))
        g.add("duplicated", g.syms(pool, k), r.integers(1, 4, k) * int(r.choice([1, 3, 1000])))
        # counts ascending / descending in symbol order: the median-of-three branches and the checksort shortcut
        k = int(r.integers(3, kmax + 1))
        s = np.sort(g.syms(pool, k))
        c = np.sort(r.integers(1, top(k) + 2, k))
        g.add("ascending", s, c)
        g.add("descending", s, c[::-1])
        g.add("strictly_ascending", s, np.arange(1, k + 1) * int(r.integers(1, 50)))
        c2 = c.copy()
        i = int(r.integers(0, k - 1))
        c2[i], c2[i + 1] = c2[i + 1], c2[i]
        g.add("nearly_sorted", s, c2)
        # Fibonacci / powers of two over 20-40 symbols: deep cuts by the 16-bit limit, symbol == package ties
        k = int(r.integers(min(20, kmax), min(40, kmax) + 1))
        f = np.array(_fib(k), np.int64)
        s = g.syms(pool, k)
        g.add("fibonacci", s, f)
        g.add("fibonacci_sorted_syms", np.sort(s), f)
        g.add("fibonacci_shuffled", s, r.permutation(f))
        k = int(r.integers(min(20, kmax), min(29, kmax) + 1))
        g.add("pow2", g.syms(pool, k), 2 ** r.permutation(k).astype(np.int64))
        g.add("pow2_ascending", np.sort(g.syms(pool, k)), 2 ** np.arange(k, dtype=np.int64))


def generate(seed: int = 2024):
    """Returns (dc, ac): lists of (kind, hist[256] uint32).  dc histograms only use symbols 0..15 (what a DC code table
    holds); ac histograms use any byte value."""
    g = _Gen(seed)
    r = g.rng
    _families(g, DC_SYMBOLS, 16, 45)
    for k in range(2, 17):
        g.add("equal_all_k", DC_SYMBOLS[:k], np.full(k, int(r.integers(1, 10 ** 6))))
    g.add("fibonacci_16", DC_SYMBOLS, _fib(16))
    g.add("fibonacci_16_rev", DC_SYMBOLS, _fib(16)[::-1])
    while len(g.out) < 1000:  # random DC-like tables: geometric over the sizes
        k = int(r.integers(1, 17))
        c = np.maximum(1, (10 ** r.uniform(2, 8)) * 0.5 ** (np.arange(k) * r.uniform(0.2, 2))).astype(np.int64)
        g.add("dc_geometric", np.sort(g.syms(DC_SYMBOLS, k)), c)
    dc = g.out[:1000]

    g.out = []
    _families(g, np.arange(256), 256, 14)
    for k in range(2, 257):  # all counts equal for every k = 2 .. 256
        g.add("equal_all_k", g.syms(np.arange(256), k), np.full(k, int(r.choice([1, 5, 4096, 10 ** 6]))))
    g.add("fibonacci_40", np.arange(40), _fib(40))
    g.add("fibonacci_43", np.arange(43), _fib(43))  # the longest Fibonacci run whose package sums stay < 2^31
    g.add("pow2_29", np.arange(29) * 7, 2 ** np.arange(29, dtype=np.int64))
    for total in (10 ** 3, 10 ** 5, 10 ** 7, 10 ** 8):  # all 256 byte values
        g.add("all256_random", np.arange(256), g.scale(r.integers(1, 1000, 256), total))
        g.add("all256_zipf", r.permutation(256), g.scale(1.0 / np.arange(1, 257) ** 1.3, total))
    g.add("all256_equal", np.arange(256), np.full(256, 3))
    g.add("all256_one_big", np.arange(256), np.r_[10 ** 8, np.ones(255, np.int64)])
    while len(g.out) < 1000:  # Zipf-like tables over the 162 real AC symbols, totals up to 10^8
        k = int(r.integers(20, 163))
        z = 1.0 / np.arange(1, k + 1) ** r.uniform(0.6, 2.5)
        g.add("ac_zipf", g.syms(AC_SYMBOLS, k), g.scale(z, 10 ** r.uniform(3, 8)))
    ac = g.out[:1000]
    return dc, ac


# ---- plain references, written for the tests (not ports of the table builders) -------------------------------------

def optimal_cost(counts, max_len: int = MAX_LEN) -> int:
    """Least sum of count * length over prefix codes of length <= max_len for the counts plus one zero-count leaf:
    the textbook package-merge (coin collector) over Python lists of weights."""
    leaves = sorted([int(c) for c in counts] + [0])
    n = len(leaves)
    if n == 1:
        return 0
    cur = list(leaves)
    for _ in range(max_len - 1):
        pk = [cur[2 * i] + cur[2 * i + 1] for i in range(len(cur) // 2)]
        cur = sorted(leaves + pk)
    return sum(cur[: 2 * n - 2])


def canonical_codes(bits, vals):
    """{symbol: (code, length)} as a JPEG decoder reads BITS / HUFFVAL (ff_mjpeg_build_huffman_codes)."""
    out, code, k = {}, 0, 0
    for length in range(1, 17):
        for _ in range(bits[length]):
            out[int(vals[k])] = (code, length)
            code += 1
            k += 1
        code <<= 1
    return out


def code_table_entry(sym: int, code: int, length: int) -> int:
    """K4a's code-table word: the code shifted over the symbol's nb = sym & 15 mantissa bits, then (code << nb) << 5 |
    (length + nb), as a 32-bit value (a real AC symbol has nb <= 10, so nothing is lost there)."""
    nb = sym & 15
    return (((code << nb) << 5) | (length + nb)) & 0xFFFFFFFF


def dht_segment(bits4, vals4, nvals4) -> bytes:
    """The DHT segment of a picture header (mjpegenc_common.c): the four tables DC0, DC1, AC0, AC1."""
    body = b""
    for t in range(4):
        body += bytes([((t >> 1) << 4) | (t & 1)]) + bytes(int(b) for b in bits4[t][1:17]) + bytes(int(v) for v in vals4[t][: nvals4[t]])
    return b"\xff\xc4" + (len(body) + 2).to_bytes(2, "big") + body


def check_table(hist, bits, vals, nvals):
    """Properties of a table built from `hist` that do not depend on tie order.  Returns a list of what is wrong."""
    hist = [int(x) for x in hist]
    used = [s for s in range(256) if hist[s]]
    bad = []
    if nvals != len(used):
        return [f"nvals {nvals} != {len(used)} used symbols"]
    if int(bits[0]) != 0 or sum(int(b) for b in bits[1:17]) != nvals:
        return [f"sum BITS {sum(int(b) for b in bits[1:17])} != nvals {nvals} (bits[0] = {int(bits[0])})"]
    if sorted(int(v) for v in vals[:nvals]) != used:
        return ["HUFFVAL is not a permutation of the used symbols"]
    codes = canonical_codes(bits, vals)
    length = {s: codes[s][1] for s in used}
    kraft = sum(1 << (MAX_LEN - l) for l in length.values())
    if kraft >= 1 << MAX_LEN:
        bad.append(f"Kraft sum {kraft} / 2^16 is not < 1 (the all-ones code must stay free)")
    shortest_below = None  # shortest length among the symbols with a smaller count
    for c in sorted(set(hist[s] for s in used)):
        group = [length[s] for s in used if hist[s] == c]
        if shortest_below is not None and max(group) > shortest_below:
            bad.append(f"count {c} got length {max(group)}, longer than {shortest_below} of a smaller count")
            break
        shortest_below = min(group) if shortest_below is None else min(shortest_below, min(group))
    cost = sum(hist[s] * length[s] for s in used)
    opt = optimal_cost([hist[s] for s in used])
    if cost != opt:
        bad.append(f"sum count*length {cost} != optimum {opt}")
    return bad
