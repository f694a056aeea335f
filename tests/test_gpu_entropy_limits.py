"""Frames at the entropy coder's limits, end to end against the CPU oracle, at qscale 1 and in all three chroma formats.

The frames are put together from a library of 8x8 blocks whose quantised levels the oracle's FDCT and quantiser
(orc_fdct_sse2, orc_quantize) give: cosine-basis and 0/255 sign patterns of one DCT basis function at swept amplitudes.
  * the coverage frame holds every (run, size) symbol the encoder can emit, in both signs, ZRL chains (runs of exactly 15,
    16, 32 and 48) and a block whose only AC level sits at zigzag position 63 (three ZRLs, then (14, s), and no EOB);
  * the deep-code frames are mostly flat, with single-level blocks in a Fibonacci spread of counts and size-9 symbols
    once per table: those get 16-bit codes, so their code-table entries use all 32 bits and K4a puts 25-bit items.  One
    frame per K4a path: such items in a block of K4a's 256-bit slot path, in a block of more than 256 bits (emitted
    straight into the warp's window) and in a 32-block unit of more than 8 Kibit (the clipped, windowed path).
Every test asserts that the feature it targets is present, so that it cannot silently stop exercising it."""
import functools

import numpy as np
import pytest

from tests.support import histograms as H
from tests.support.scan_model import block_bits, coding_order, frame_from_blocks

pytestmark = pytest.mark.gpu

QSCALE = 1
W = 512  # 32 MCUs per row at 4:2:0 / 4:2:2: two K2 tiles of 16 MCUs, none wraps a row


@functools.lru_cache(maxsize=None)
def _tools():
    from tests.support import oracle as orc

    lib = orc.oracle()
    im, q16, b16 = np.zeros(64, np.uint8), np.zeros(64, np.uint16), np.zeros(64, np.uint16)
    lib.orc_build_matrices(QSCALE, im.ctypes.data, q16.ctypes.data, b16.ctypes.data)
    c = np.array([[np.cos((2 * i + 1) * u * np.pi / 16) for i in range(8)] for u in range(8)])
    basis = [np.outer(c[orc.ZIGZAG[p] // 8], c[orc.ZIGZAG[p] % 8]) for p in range(64)]
    return orc, lib, q16, b16, basis


def levels(px):
    """quantised levels (zigzag order) of one 8x8 block of pixels at QSCALE"""
    orc, lib, q16, b16, _ = _tools()
    b = np.ascontiguousarray(px.reshape(64).astype(np.int16))
    lib.orc_fdct_sse2(b.ctypes.data)
    zz = np.zeros(64, np.int16)
    lib.orc_quantize(b.ctypes.data, zz.ctypes.data, q16.ctypes.data, b16.ctypes.data)
    return zz


def block(terms, base=128.0):
    """128 + a sum of DCT basis functions (zigzag position p, amplitude a, as a cosine or as its 0/255-like sign pattern)"""
    basis = _tools()[4]
    f = np.full((8, 8), base)
    for p, a, square in terms:
        f += a * (np.sign(basis[p]) if square else basis[p] / np.abs(basis[p]).max())
    return np.clip(np.round(f), 0, 255).astype(np.uint8)


def ac_symbols(zz):
    """(symbol, level) of a block's AC part as the encoder records them (mjpegenc.c): ZRLs, (run << 4) | size, EOB"""
    out, run = [], 0
    nz = np.nonzero(zz[1:])[0]
    last = int(nz[-1]) + 1 if nz.size else 0
    for i in range(1, last + 1):
        v = int(zz[i])
        if v == 0:
            run += 1
            continue
        while run >= 16:
            out.append((0xF0, 0))
            run -= 16
        out.append(((run << 4) | abs(v).bit_length(), v))
        run = 0
    if last < 63:
        out.append((0x00, 0))
    return out


@functools.lru_cache(maxsize=None)
def library():
    """{block pixels (bytes): AC symbols} of single-basis blocks over every position, amplitude, sign and shape"""
    amps = np.concatenate([np.arange(1, 20, 0.5), np.arange(20, 128, 1.0), [127.5, 140, 170, 200, 255]])
    out = []
    for p in range(1, 64):
        for square in (False, True):
            for a in amps:
                for sgn in (1, -1):
                    px = block([(p, sgn * a, square)])
                    out.append((px, ac_symbols(levels(px))))
    return out


def max_ac_size():
    """the largest AC size at QSCALE: a 0/255 sign pattern of one basis function maximises that coefficient"""
    return max(abs(int(v)).bit_length() for px, syms in library() for _, v in syms)


def coverage_blocks():
    """one block per (run, size, sign) the encoder can emit, plus the ZRL chain blocks"""
    want = {}
    for px, syms in library():
        for s, v in syms:
            if s not in (0x00, 0xF0):
                want.setdefault((s, v > 0), px)
    chains = {}
    for r in (15, 16, 32, 48):  # a level at position 1, then one after exactly r zeros
        chains[r] = _two_level_block(1, 1 + r + 1)
    # one level at position 63 and nothing else: three ZRLs, (14, s), no EOB
    last = next(px for px, syms in library() if [s for s, _ in syms][:3] == [0xF0] * 3 and len(syms) == 4 and syms[3][0] >> 4 == 14)
    return want, chains, last


def _two_level_block(q, p):
    for a in (8, 12, 16, 24, 32):
        for b in (8, 12, 16, 24, 32, 48):
            px = block([(q, a, False), (p, b, False)])
            zz = levels(px)
            if zz[q] and zz[p] and not zz[1:q].any() and not zz[q + 1: p].any():
                return px
    raise AssertionError(f"no block with levels at {q} and {p} only")


def single_level(sym):
    """a block whose AC part is exactly one level coded with `sym`, then EOB"""
    for px, syms in library():
        if len(syms) == 2 and syms[0][0] == sym and syms[1][0] == 0:
            return px
    raise AssertionError(hex(sym))


def heavy_block(rng, base=None, first=1):
    """base (flat by default) plus every basis function from zigzag position `first` on at one small amplitude and a random
    sign: all those levels non-zero, sizes 2 to 5, so the block needs well over 256 bits while its AC symbols are the few
    (0, size) ones, frequent in any frame that has such blocks"""
    basis = _tools()[4]
    base = block([]) if base is None else base
    for _ in range(100):
        f = base.astype(np.float64)
        for k in range(first, 64):
            f = f + float(rng.choice([-1, 1])) * 6.0 * basis[k] / np.abs(basis[k]).max()
        px = np.clip(np.round(f), 0, 255).astype(np.uint8)
        zz = levels(px)
        if (zz[:first] == levels(base)[:first]).all() and zz[first:].all():
            return px
    raise AssertionError("no heavy block found")


def _planes(chroma_format, luma_blocks, chroma_blocks, h):
    """planes of a W x h frame: the given blocks in raster block order from the top left, flat (128) elsewhere.
    chroma_blocks = (Cb blocks, Cr blocks)"""
    orc = _tools()[0]
    ch, cw = orc.chroma_shape(W, h, chroma_format)
    y = np.full((h, W), 128, np.uint8)
    cb, cr = np.full((ch, cw), 128, np.uint8), np.full((ch, cw), 128, np.uint8)
    for plane, blocks in ((y, luma_blocks), (cb, chroma_blocks[0]), (cr, chroma_blocks[1])):
        per_row = plane.shape[1] // 8
        assert len(blocks) <= per_row * (plane.shape[0] // 8), "frame too small for its blocks"
        for k, px in enumerate(blocks):
            by, bx = divmod(k, per_row)
            plane[8 * by: 8 * by + 8, 8 * bx: 8 * bx + 8] = px
    return y, cb, cr


def coverage_frame(chroma_format):
    want, chains, last = coverage_blocks()
    blocks = list(want.values()) + list(chains.values()) + [last]
    return _planes(chroma_format, blocks, (blocks, blocks[::-1]), 256)


FIB_SYMBOLS = [0x12, 0x13, 0x23, 0x32, 0x14, 0x24, 0x33, 0x43, 0x52, 0x62, 0x72, 0x82, 0x34, 0x44, 0x53, 0x63]
DEEP = (0x99, 0xD9)  # size 9 after runs of 9 and 13


PATHS = ("slot", "direct", "clip")


def deep_frame(chroma_format, path, h=1536):
    """A frame whose size-9 symbols of DEEP get 16-bit codes in both AC tables, so that their code-table entries use all 32
    bits and K4a puts 25-bit items, on one K4a path per frame (a unit is 32 consecutive blocks in coding order):
      slot:   DEEP once per table in single-level blocks (a block of <= 256 bits);
      direct: DEEP[0] once per table in a heavy block (> 256 bits) of a unit that stays below 8 Kibit;
      clip:   DEEP[0] once per table in a unit of heavy blocks only (> 8 Kibit).
    The rest is flat but for single-level blocks whose counts make a Fibonacci spread in each table: that, and the heavy
    blocks using only a few frequent symbols, keeps the tree 16 levels deep under DEEP."""
    rng = np.random.default_rng(9 + PATHS.index(path))
    order = coding_order(chroma_format, W, h)
    cls = [min(pl, 1) for pl, _, _ in order]
    deep = [single_level(s) for s in DEEP]
    pos0 = next(p for p in range(1, 64) if levels(deep[0])[p])
    blocks = [None] * len(order)
    start = 64  # units 0 and 1 stay flat
    if path == "slot":
        features = {0: deep, 1: deep}
    elif path == "direct":
        features = {c: [heavy_block(rng, deep[0], pos0 + 1)] for c in (0, 1)}
    else:
        for i in range(start, start + 32):
            blocks[i] = heavy_block(rng)
        for c in (0, 1):
            blocks[next(i for i in range(start + 8, start + 32) if cls[i] == c)] = heavy_block(rng, deep[0], pos0 + 1)
        start += 32
        features = {0: [], 1: []}
    spread, f = [], [1, 2]
    while len(f) < len(FIB_SYMBOLS):
        f.append(f[-1] + f[-2])
    for s, n in zip(FIB_SYMBOLS, f):
        spread += [single_level(s)] * n
    if path != "slot":
        # heavy blocks alone in each of the frame's last 64 units: their (0, size) symbols become frequent, not rare ones that
        # would sit under DEEP in the tree
        for k in range(1, 65):
            blocks[len(order) - 32 * k + k % 8] = heavy_block(rng)  # (both classes, in every format)
    for c in (0, 1):  # the features first (in the unit behind `start`), then the spread, in this class's blocks
        todo = features[c] + spread
        at = [i for i in range(start, len(order)) if cls[i] == c and blocks[i] is None]
        assert len(at) >= len(todo), "frame too small for the spread"
        for i, px in zip(at, todo):
            blocks[i] = px
    return frame_from_blocks(chroma_format, W, h, blocks)


def _lengths(dbg, t):
    return {s: l for s, (c, l) in H.canonical_codes(dbg.bits[t], dbg.vals[t]).items()}


def _encode_and_compare(orc, y, u, v, chroma_format):
    """the GPU path against the oracle, as test_gpu_parity._compare does, plus an independent entropy decode of the GPU
    JPEG; returns (jpeg, oracle debug record, coefficients in coding order)"""
    import h2j_b200

    h, w = y.shape
    want, dbg, coefs = orc.oracle_encode(y, u, v, fixed_qscale=QSCALE, want_coefs=True, chroma_format=chroma_format)
    frames = np.concatenate([y.reshape(-1), u.reshape(-1), v.reshape(-1)])[None, :].copy()
    with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=1, n_slots=1, fixed_qscale=QSCALE, max_jpeg_bytes=8 << 20,
                          chroma_format=chroma_format) as e:
        e.submit_host(0, frames.ctypes.data, frames.shape[1], 1, w, h)
        res = e.collect(0)
        info = e.frame_info(0, 0)
        got_coefs = e.coefficients(0, 0, coefs.shape[0])
    bad = np.nonzero((got_coefs != coefs).any(axis=1))[0]
    assert bad.size == 0, f"{bad.size} blocks differ, first {bad[:5]}"
    for t in range(4):
        assert list(info.hist[t]) == list(dbg.hist[t]), f"histogram {t}"
        assert info.nvals[t] == dbg.nvals[t]
        assert bytes(info.bits[t]) == bytes(dbg.bits[t]), f"BITS {t}"
        assert bytes(info.vals[t])[: info.nvals[t]] == bytes(dbg.vals[t])[: dbg.nvals[t]], f"HUFFVAL {t}"
    assert info.header_bytes == dbg.header_bytes
    assert info.scan_bits == dbg.scan_bits
    assert res.status == [0]
    got = res.jpegs[0]
    assert got == want
    decoded, _ = orc.decode_coefs(got)
    assert (decoded == coefs).all()
    return got, dbg, coefs


FORMATS = [0, 1, 2]  # 4:2:0, and entropy_walk_kernel<kFmt422>, <kFmt444>


def test_max_ac_size_is_nine():
    assert max_ac_size() == 9


@pytest.mark.parametrize("chroma_format", FORMATS)
def test_every_symbol_both_signs_and_zrl_chains(orc, chroma_format):
    y, u, v = coverage_frame(chroma_format)
    _, dbg, coefs = _encode_and_compare(orc, y, u, v, chroma_format)
    per_block = [ac_symbols(z) for z in coefs]
    seen = {(s, lv > 0) for syms in per_block for s, lv in syms if s not in (0x00, 0xF0)}
    every = {((r << 4) | sz, pos) for r in range(16) for sz in range(1, max_ac_size() + 1) for pos in (True, False)}
    assert every <= seen, sorted(every - seen)[:8]
    runs = set()
    for z in coefs:
        nz = np.nonzero(z[1:])[0] + 1
        runs |= {int(b - a - 1) for a, b in zip(nz, nz[1:])}
    assert {15, 16, 32, 48} <= runs
    # a block whose only AC level is at position 63: three ZRLs, (14, s), no EOB
    assert any([s >> 4 for s, _ in syms] == [15, 15, 15, 14] for syms in per_block)


def test_coding_order_matches_the_encoder(orc):
    rng = np.random.default_rng(3)
    for fmt in FORMATS:
        n = len(coding_order(fmt, W, 32))
        blocks = [rng.integers(0, 256, (8, 8)).astype(np.uint8) for _ in range(n)]
        _, _, coefs = orc.oracle_encode(*frame_from_blocks(fmt, W, 32, blocks), fixed_qscale=QSCALE, want_coefs=True, chroma_format=fmt)
        assert all((coefs[i][1:] == levels(px)[1:]).all() for i, px in enumerate(blocks)), fmt


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("chroma_format", FORMATS)
def test_25_bit_items_on_every_k4a_path(orc, chroma_format, path):
    """Size-9 symbols with 16-bit codes (25-bit items) in both AC tables, on K4a's slot path (a block of <= 256 bits in a
    unit of <= 8 Kibit), direct path (a block of > 256 bits in such a unit) or clipped windowed path (a unit of > 8 Kibit)."""
    h = 1536
    y, u, v = deep_frame(chroma_format, path, h)
    _, dbg, coefs = _encode_and_compare(orc, y, u, v, chroma_format)
    for t in (2, 3):
        L = _lengths(dbg, t)
        assert L[DEEP[0]] == 16 and (path != "slot" or L[DEEP[1]] == 16), (t, {hex(s): L.get(s) for s in DEEP})
    bits, classes = block_bits(dbg, coefs, chroma_format, W, h)
    assert sum(bits) == dbg.scan_bits
    unit_bits = [sum(bits[i: i + 32]) for i in range(0, len(bits), 32)]  # entropy_walk_kernel: unit u = blocks 32u .. 32u + 31
    seen = set()
    for i, z in enumerate(coefs):
        if any(s in DEEP for s, _ in ac_symbols(z)):
            where = "clip" if unit_bits[i // 32] > 8192 else ("direct" if bits[i] > 256 else "slot")
            seen.add((where, classes[i]))
    assert seen == {(path, 0), (path, 1)}, seen
