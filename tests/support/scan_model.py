"""What the last two stages of the pipeline must produce, derived from the CPU oracle alone, and frames that put those
stages at their boundaries.

K4b (scan_place_kernel) joins the staged units -- 32 consecutive blocks in coding order -- into one bit stream: unit u
starts at bit P[u] of the scan, carries c = P & 31 bits of an incomplete word in from the unit in front, and emits the
(c + its length) >> 5 words it completes.  A group of 256 units finds its offset by a look-back; inside a group a warp
concatenates a run of 8 or 32 units, and only a run's first unit reads its carry from the staged tail of the unit in
front -- from two staged words (`hiw`) when that unit's last word holds fewer than c bits.  The frame's last word is
padded with ones to a byte.  K4b also counts the 0xFF bytes of every 1024-word chunk; K5 (stuff_kernel) places chunk k
from the counts in front of it, at byte a0 = (header bytes + 0xFF bytes in front) mod 16 of its 16-byte output line.

Everything here comes from one oracle encode: the unstuffed scan is the JPEG's bytes from header_bytes up to EOI with
the 0x00 behind every 0xFF dropped, and the unit lengths are the oracle's coefficients coded with its Huffman tables.
Each case builder searches seeded frames until its edge is present (deterministically, cached).  TEST INFRASTRUCTURE
ONLY."""
from __future__ import annotations

import functools
from dataclasses import dataclass
from typing import Callable, Iterable, Optional, Tuple

import numpy as np

from tests.support import histograms as H
from tests.support import oracle as orc

UNIT_BLOCKS = 32     # blocks per K4a unit
GROUP_UNITS = 256    # units per K4b group
CHUNK_WORDS = 1024   # K4b counts 0xFF bytes, and K5 works, per 1024 scan words
CHUNK_BYTES = 4 * CHUNK_WORDS
QSCALE = 2


def coding_order(chroma_format, w, h):
    """(plane, block row, block column) of every block of a w x h frame (whole MCUs: w and h multiples of 16) in the order
    the encoder codes them (mjpegenc.c ff_mjpeg_encode_mb, see oracle/mjpeg_oracle.c): plane 0 is Y, 1 Cb, 2 Cr"""
    assert w % 16 == 0 and h % 16 == 0, "whole MCUs only"
    out = []
    for my in range(h // 16):
        for mx in range(w // 16):
            y = [(0, 2 * my + r, 2 * mx + c) for r in range(2) for c in range(2)]
            if chroma_format == 0:
                out += y + [(1, my, mx), (2, my, mx)]
            elif chroma_format == 1:
                out += y + [(1, 2 * my, mx), (1, 2 * my + 1, mx), (2, 2 * my, mx), (2, 2 * my + 1, mx)]
            else:  # two 8x16 MCUs per macroblock, every component 1x2
                for c in range(2):
                    out += [(pl, 2 * my + r, 2 * mx + c) for pl in range(3) for r in range(2)]
    return out


def frame_from_blocks(chroma_format, w, h, blocks):
    """planes of a w x h frame whose coded blocks are blocks[i] (coding order; None or missing: flat)"""
    ch, cw = orc.chroma_shape(w, h, chroma_format)
    planes = [np.full((h, w), 128, np.uint8), np.full((ch, cw), 128, np.uint8), np.full((ch, cw), 128, np.uint8)]
    order = coding_order(chroma_format, w, h)
    assert len(blocks) <= len(order), "frame too small for its blocks"
    for (pl, r, c), px in zip(order, blocks):
        if px is not None:
            planes[pl][8 * r: 8 * r + 8, 8 * c: 8 * c + 8] = px
    return tuple(planes)


@functools.lru_cache(maxsize=None)
def block_index(chroma_format, w, h):
    """per plane, the coding-order index of the block every pixel belongs to"""
    ch, cw = orc.chroma_shape(w, h, chroma_format)
    idx = [np.zeros((h // 8, w // 8), np.int64), np.zeros((ch // 8, cw // 8), np.int64), np.zeros((ch // 8, cw // 8), np.int64)]
    for i, (pl, r, c) in enumerate(coding_order(chroma_format, w, h)):
        idx[pl][r, c] = i
    return tuple(np.kron(p, np.ones((8, 8), np.int64)) for p in idx)


def _length_table(dbg, t):
    out = np.full(256, 1 << 20, np.int64)  # a symbol without a code makes any sum absurd
    for s, (_, n) in H.canonical_codes(dbg.bits[t], dbg.vals[t]).items():
        out[s] = n
    return out


def _bit_length(x):
    return np.frexp(np.abs(x).astype(np.float64))[1].astype(np.int64)


def block_bits(dbg, coefs, chroma_format, w, h):
    """bits K4a emits for every block in coding order, from the oracle's tables; and the class (0 luma, 1 chroma) of each"""
    dc_len, ac_len = [_length_table(dbg, 0), _length_table(dbg, 1)], [_length_table(dbg, 2), _length_table(dbg, 3)]
    plane = np.array([pl for pl, _, _ in coding_order(chroma_format, w, h)], np.int64)
    cls = np.minimum(plane, 1)
    z = coefs.astype(np.int64)
    diff = np.zeros(len(z), np.int64)
    for pl in range(3):  # mjpegenc's DC predictors start at 128 (1024 >> 3)
        at = np.flatnonzero(plane == pl)
        dc = z[at, 0]
        diff[at] = dc - np.concatenate([[128], dc[:-1]])
    size = _bit_length(diff)
    bits = np.where(cls == 0, dc_len[0][size], dc_len[1][size]) + size
    ac = z[:, 1:]
    pos = np.arange(1, 64)
    nz = ac != 0
    last = np.maximum.accumulate(np.where(nz, pos, 0), axis=1)
    prev = np.concatenate([np.zeros((len(z), 1), np.int64), last[:, :-1]], axis=1)  # the non-zero level before each position
    run = pos - prev - 1
    s = _bit_length(ac)
    sym = ((run & 15) << 4) | s
    for c in (0, 1):
        L = ac_len[c]
        per = np.where(nz, L[sym] + s + (run >> 4) * L[0xF0], 0).sum(axis=1) + np.where(last[:, -1] < 63, L[0x00], 0)
        bits = bits + np.where(cls == c, per, 0)
    return bits.tolist(), cls.tolist()


def unstuff(stuffed: bytes) -> np.ndarray:
    """the scan with the 0x00 behind every 0xFF dropped (every 0xFF must have one)"""
    b = np.frombuffer(stuffed, np.uint8)
    ff = np.flatnonzero(b == 0xFF)
    assert ff.size == 0 or (ff[-1] + 1 < b.size and not b[ff + 1].any()), "a 0xFF without its stuffed 0x00"
    keep = np.ones(b.size, bool)
    keep[ff + 1] = False
    return b[keep]


class Scan:
    """One oracle encode and the positions K4b and K5 must reproduce."""

    def __init__(self, planes, chroma_format, qscale=QSCALE, comment: Optional[bytes] = None):
        y, u, v = planes
        h, w = y.shape
        self.jpeg, self.dbg, self.coefs = orc.oracle_encode(y, u, v, fixed_qscale=qscale, comment=comment, want_coefs=True,
                                                            chroma_format=chroma_format)
        self.header_bytes, self.scan_bits = int(self.dbg.header_bytes), int(self.dbg.scan_bits)
        bits, _ = block_bits(self.dbg, self.coefs, chroma_format, w, h)
        bits = np.asarray(bits, np.int64)
        self.n_blocks = bits.size
        self.n_units = -(-bits.size // UNIT_BLOCKS)
        self.unit_bits = np.add.reduceat(bits, np.arange(0, bits.size, UNIT_BLOCKS))
        assert self.unit_bits.sum() == self.scan_bits, "unit lengths do not add up to the oracle's scan"
        self.start = np.concatenate([[0], np.cumsum(self.unit_bits)[:-1]])  # P: each unit's first bit
        self.carry = self.start & 31                                           # c: bits it carries in
        self.words = (self.carry + self.unit_bits) >> 5                        # output words it completes
        self.last_word_bits = ((self.unit_bits - 1) & 31) + 1                  # bits of its last staged word
        # the carry of unit u spans the last two staged words of unit u - 1
        self.hiw = np.zeros(self.n_units, bool)
        self.hiw[1:] = (self.carry[1:] != 0) & (self.last_word_bits[:-1] < self.carry[1:])
        self.group_start = self.start[::GROUP_UNITS]
        assert self.jpeg[-2:] == b"\xff\xd9"
        self.data = unstuff(self.jpeg[self.header_bytes: -2])
        self.n_bytes = self.data.size
        assert self.n_bytes == (self.scan_bits + 7) // 8
        self.ff = np.flatnonzero(self.data == 0xFF)
        self.stuffed_ff = int(self.ff.size)
        self.n_words = -(-self.n_bytes // 4)
        self.n_chunks = -(-self.n_words // CHUNK_WORDS)
        self.chunk_ff = np.bincount(self.ff // CHUNK_BYTES, minlength=self.n_chunks)
        self.chunk_ff_before = np.concatenate([[0], np.cumsum(self.chunk_ff)[:-1]])
        self.a0 = (self.header_bytes + self.chunk_ff_before) % 16  # K5's offset of each chunk in its 16-byte output line

    @property
    def groups(self):
        return -(-self.n_units // GROUP_UNITS)

    def run_starts(self, upw):
        """units that begin a run of `upw` inside a group (not a group's first unit)"""
        u = np.arange(upw, self.n_units, upw)
        return u[u % GROUP_UNITS != 0]


# ---- the edges --------------------------------------------------------------------------------------------------------

def _group_firsts(s):
    return np.arange(GROUP_UNITS, s.n_units, GROUP_UNITS)


def _run_start_edge(upw):
    def edge(s):
        u = s.run_starts(upw)
        u = u[u % (4 * upw) != 0] if upw == 8 else u  # 8: not also a 32-unit boundary
        c = s.carry[u] != 0
        return bool((c & s.hiw[u]).any() and (c & ~s.hiw[u]).any())
    return edge


def _aligned_unit(s):
    u = np.arange(s.n_units - 1)
    return bool(((s.unit_bits[u] % 32 == 0) & ((u + 1) % 8 == 0) & (s.carry[u + 1] != 0)).any())


def _chunk_end_ffs(s):
    k = np.arange(1, s.n_chunks) * CHUNK_BYTES
    return bool((s.data[k - 1] == 0xFF).any() and (s.data[k] == 0xFF).any())


def _zero_chunk(s):
    k = np.arange(1, s.n_chunks - 1)
    return bool(((s.chunk_ff[k] == 0) & (s.chunk_ff[k + 1] > 0) & (s.chunk_ff_before[k] > 0)).any())


EDGES: dict[str, Callable[[Scan], bool]] = {
    # K4b
    "group_first_c0": lambda s: bool((s.carry[_group_firsts(s)] == 0).any()),
    "group_first_hiw": lambda s: bool(s.hiw[_group_firsts(s)].any()),
    "run8_first_carry": _run_start_edge(8),
    "run32_first_carry": _run_start_edge(32),
    "unit_bits_multiple_of_32": _aligned_unit,
    "unit_words": lambda s: bool({32, 63, 64} <= set(s.words.tolist()) and (s.words > 96).any()),
    "units_255": lambda s: s.n_units == 255,
    "units_256": lambda s: s.n_units == 256,
    "units_257": lambda s: s.n_units == 257,
    "units_512": lambda s: s.n_units == 512,
    "units_513": lambda s: s.n_units == 513,
    # the frame's end
    "end_word_aligned": lambda s: s.scan_bits % 32 == 0,
    "end_byte_aligned": lambda s: s.scan_bits % 8 == 0 and s.scan_bits % 32 != 0,
    "padding_makes_ff": lambda s: s.scan_bits % 8 != 0 and s.data[-1] == 0xFF,
    **{f"bytes_mod16_{r}": (lambda r: lambda s: s.n_bytes % 16 == r)(r) for r in range(16)},
    "bytes_4096": lambda s: s.n_bytes == CHUNK_BYTES,
    "bytes_4097": lambda s: s.n_bytes == CHUNK_BYTES + 1,
    "bytes_8192": lambda s: s.n_bytes == 2 * CHUNK_BYTES,
    "bytes_8193": lambda s: s.n_bytes == 2 * CHUNK_BYTES + 1,
    # K5
    "ff_at_chunk_ends": _chunk_end_ffs,
    "zero_chunk_before_counts": _zero_chunk,
    "chunks_1": lambda s: s.n_chunks == 1,
    "chunks_32": lambda s: s.n_chunks == 32,
    "chunks_over_64": lambda s: s.n_chunks > 64,  # every K5 CTA of the frame takes three chunks or more
}
K4B_EDGES = [k for k in EDGES if k.startswith(("group", "run", "unit"))]
SIZE_EDGES = [k for k in EDGES if k.startswith("units_")]
END_EDGES = [k for k in EDGES if k.startswith(("end_", "padding", "bytes_"))]
K5_EDGES = [k for k in EDGES if k.startswith(("ff_", "zero_", "chunks_"))]
# the edges also built at 4:2:2 and 4:4:4
FORMAT_EDGES = ["group_first_c0", "group_first_hiw", "run8_first_carry", "run32_first_carry", "end_word_aligned", "padding_makes_ff",
                "ff_at_chunk_ends"]


# ---- frame families ---------------------------------------------------------------------------------------------------

def geometry_for_units(n_units, chroma_format):
    """the most square whole-MCU frame with exactly n_units units"""
    best = None
    for mw in range(1, 200):
        for mh in range(1, 200):
            n = -(-orc.blocks_of(16 * mw, 16 * mh, chroma_format) // UNIT_BLOCKS)
            if n == n_units and (best is None or abs(mw - mh) < abs(best[0] - best[1])):
                best = (mw, mh)
    assert best, n_units
    return 16 * best[0], 16 * best[1]


def textured(chroma_format, w, h, seed, amp=30):
    return orc.synth_planes_fmt(w, h, chroma_format, "textured", seed=seed, amp=amp)


def noise(chroma_format, w, h, seed, amp=30):
    return orc.synth_planes_fmt(w, h, chroma_format, "noise", seed=seed, amp=amp)


def ramp(chroma_format, w, h, seed, lo=0, hi=16):
    """noise whose amplitude grows from lo to hi down the frame: unit lengths over a wide range"""
    out = []
    for k, p in enumerate(noise(chroma_format, w, h, seed, amp=1)):
        rng = np.random.default_rng(seed * 3 + k)
        a = np.linspace(lo, hi, p.shape[0])[:, None]
        out.append(np.clip(np.round(128 + a * rng.uniform(-1, 1, p.shape)), 0, 255).astype(np.uint8))
    return tuple(out)


def flat_band(chroma_format, w, h, seed, top, bottom):
    """textured frame, flat (128) from row `top` to row `bottom` (luma rows, multiples of 16): a stretch of the scan without
    0xFF bytes between two with many"""
    y, u, v = textured(chroma_format, w, h, seed, amp=60)
    vs = 2 if chroma_format == 0 else 1
    y[top:bottom] = 128
    u[top // vs: bottom // vs] = 128
    v[top // vs: bottom // vs] = 128
    return y, u, v


def partial_noise(chroma_format, w, h, seed, m, amp=40, tail=None):
    """blocks [0, m) in coding order noise of amplitude amp, the rest flat; tail = (fraction, pixels, seed) makes block m
    noise of amp * fraction in that many of its pixels: a frame's scan length is set to the byte this way"""
    idx = block_index(chroma_format, w, h)
    out = []
    for k, (p, ix) in enumerate(zip(noise(chroma_format, w, h, seed, amp=amp), idx)):
        q = np.where(ix < m, p, 128).astype(np.uint8)
        if tail is not None:
            frac, npx, ts = tail
            at = np.flatnonzero(ix.reshape(-1) == m)
            if at.size:
                rng = np.random.default_rng(ts * 7 + k)
                pick = at[rng.permutation(at.size)[:npx]]
                q.reshape(-1)[pick] = np.clip(np.round(128 + frac * amp * rng.uniform(-1, 1, pick.size)), 0, 255).astype(np.uint8)
        out.append(q)
    return tuple(out)


@dataclass
class Case:
    name: str
    chroma_format: int
    planes: Tuple[np.ndarray, np.ndarray, np.ndarray]
    scan: Scan
    qscale: int = QSCALE
    comment: Optional[bytes] = None

    @property
    def size(self):
        return self.planes[0].shape[1], self.planes[0].shape[0]


def _first(name, fmt, frames: Iterable, edge=None, comment=None) -> Case:
    edge = edge or EDGES[name]
    for planes in frames:
        s = Scan(planes, fmt, comment=comment)
        if edge(s):
            return Case(name, fmt, tuple(planes), s, comment=comment)
    raise AssertionError(f"{name} (chroma format {fmt}): no frame of the search has the edge")


def _tuned(name, fmt, w, h, lo, hi, seed=0, amp=40, trials=400):
    """a partial_noise frame whose unstuffed scan has lo..hi bytes and whose edge is present: bisection over the noisy
    blocks, then seeded partial noise in the block at the step"""
    edge = EDGES[name]
    scan_at = lambda m: Scan(partial_noise(fmt, w, h, seed, m, amp), fmt)
    a, b = 0, orc.blocks_of(w, h, fmt)
    assert scan_at(b).n_bytes >= lo, "frame too small for the target"
    while a < b:  # smallest m with at least lo bytes
        m = (a + b) // 2
        if scan_at(m).n_bytes >= lo:
            b = m
        else:
            a = m + 1
    for m in (a, a - 1):
        s = scan_at(m)
        if lo <= s.n_bytes <= hi and edge(s):
            return Case(name, fmt, partial_noise(fmt, w, h, seed, m, amp), s)
    rng = np.random.default_rng(seed + 17)
    for t in range(trials):
        tail = (float(rng.uniform(0.05, 1.0)), int(rng.integers(1, 65)), t)
        planes = partial_noise(fmt, w, h, seed, a - 1, amp, tail)
        s = Scan(planes, fmt)
        if lo <= s.n_bytes <= hi and edge(s):
            return Case(name, fmt, planes, s)
    raise AssertionError(f"{name}: no tuned frame within {trials} trials")


BUILDERS: dict[str, Callable[[int], Case]] = {
    "group_first_c0": lambda f: _first("group_first_c0", f, (textured(f, 1920, 1088, s) for s in range(60))),
    "group_first_hiw": lambda f: _first("group_first_hiw", f, (textured(f, 1024, 1024, s) for s in range(20))),
    "run8_first_carry": lambda f: _first("run8_first_carry", f, (textured(f, 512, 512, s) for s in range(20))),
    "run32_first_carry": lambda f: _first("run32_first_carry", f, (textured(f, 1024, 512, s) for s in range(20))),
    "unit_bits_multiple_of_32": lambda f: _first("unit_bits_multiple_of_32", f, (textured(f, 512, 512, s) for s in range(40))),
    "unit_words": lambda f: _first("unit_words", f, (ramp(f, 1024, 1024, s) for s in range(20))),
    **{k: (lambda k: lambda f: _first(k, f, (textured(f, *geometry_for_units(int(k[6:]), f), s) for s in range(1))))(k) for k in SIZE_EDGES},
    **{k: (lambda k: lambda f: _first(k, f, (textured(f, 64, 64, s, amp=20 + s % 40) for s in range(2000))))(k)
       for k in ("end_word_aligned", "end_byte_aligned", "padding_makes_ff") + tuple(f"bytes_mod16_{r}" for r in range(16))},
    "bytes_4096": lambda f: _tuned("bytes_4096", f, 128, 128, 4096, 4096),
    "bytes_4097": lambda f: _tuned("bytes_4097", f, 128, 128, 4097, 4097),
    "bytes_8192": lambda f: _tuned("bytes_8192", f, 256, 256, 8192, 8192),
    "bytes_8193": lambda f: _tuned("bytes_8193", f, 256, 256, 8193, 8193),
    "ff_at_chunk_ends": lambda f: _first("ff_at_chunk_ends", f, (noise(f, 1024, 1024, s, amp=60) for s in range(20))),
    "zero_chunk_before_counts": lambda f: _first("zero_chunk_before_counts", f, (flat_band(f, 1024, 1024, s, 192, 832) for s in range(10))),
    "chunks_1": lambda f: _tuned("chunks_1", f, 128, 128, 3584, 4095),
    "chunks_32": lambda f: _tuned("chunks_32", f, 512, 512, 31 * CHUNK_BYTES + 1, 32 * CHUNK_BYTES),
    "chunks_over_64": lambda f: _first("chunks_over_64", f, (textured(f, 1024, 768, s) for s in range(10))),
}
assert set(BUILDERS) == set(EDGES)


@functools.lru_cache(maxsize=None)
def case(name: str, chroma_format: int = 0) -> Case:
    return BUILDERS[name](chroma_format)


COMMENT_FRAME = ("chunks_over_64", 0)  # a0 sweep: this frame under 16 comment lengths


@functools.lru_cache(maxsize=None)
def comment_case(length: int) -> Case:
    """the COMMENT_FRAME case with a COM segment of `length` characters: header_bytes grows by one per character"""
    base = case(*COMMENT_FRAME)
    text = bytes((b"abcdefghijklmnopqrstuvwxyz"[i % 26] for i in range(length)))
    return Case(f"comment_{length}", base.chroma_format, base.planes, Scan(base.planes, base.chroma_format, comment=text), comment=text)


MAX_COMMENT = 65532  # a COM segment's length field holds the text, its NUL and the field itself: 65535 at most
