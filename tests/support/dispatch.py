"""The dispatch matrix: encoder calls chosen so that every kernel the library compiles runs, at the launch shapes where
kernels go wrong, and a model of what each call launches and computes at every stage.

A case is encoder settings (chroma format, fixed_qscale, range_mode), an input path (an entry point and the way its frames
are read: in place, repitched, split, converted), the pipeline's form (batch: one layout at one stride; list: per-frame
descriptors), the FDCT kernel's tiles per CTA (0 = automatic) and the frames.  The K4b form (8 or 32 units per warp) follows
from the frames; each case is built to take the form it names.

The committed matrix is a fixed-seed covering array: every pair of values of (format, path, form, tiles, K4b form, settings)
that some valid case holds is held by some case of the matrix, plus the cases of required().  A case is valid when its
entry point can take its form (16-bit and single-picture calls have no list form; a single picture has too few K4b groups
for the 32 form) and its frames fit: sources of at most 3840x2160, at most MAX_FRAMES frames.

The model (kernels, launches, tiles_per_cta, k4b_width) restates the dispatch rules of h2j_api.cu (run_batch,
launch_pipeline); expected() gives each stage's product from the numpy input models and the CPU oracle.
TEST INFRASTRUCTURE ONLY."""
import itertools
import os
import random
import re
import subprocess
from dataclasses import dataclass, field
from typing import Tuple

import numpy as np

from tests.support import downscale, resize, rgb
from tests.support.layouts import CASES, align
from tests.support.oracle import chroma_shape

PTXAS_LOG = os.path.join(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))), "h264-h265-to-jpeg_b200", "lib",
                         "ptxas.log")
SEED = 20261022
SMS = 148        # B200: what the covering array is built for; the GPU test passes the device's count
MAX_FRAMES = 64  # per case
TILE_MCUS, UNIT_BLOCKS, GROUP_UNITS, FDCT_MIN_CTAS, MAX_TILES = 16, 32, 256, 16, 16  # h2j_common.cuh, h2j_k_entropy.cuh, h2j_k_fdct.cuh

FMTS = (0, 1, 2)
SETTINGS = tuple((q, r) for q in (0, 1, 31) for r in (0, 1))  # (fixed_qscale, range_mode)
FORMS = ("batch", "list")
TILES = (0, 1, 2, 3, 16)
K4B = (8, 32)
KINDS = ("textured", "noise", "ff", "blocks", "const", "binary")
SIZES = [(w, h) for w, h, _, _ in CASES] + [(17, 4098), (2562, 1442), (3840, 2160)]
BIG = (3840, 2160)


@dataclass(frozen=True)
class Path:
    name: str
    kind: str        # planar | sp | host | d16 | down | rgb | resize | frame | frame16 | frame_rgb | convert_pad
    aligned: bool = True
    knob: Tuple[Tuple[str, int], ...] = ()
    depth: int = 8
    factor: int = 1
    rgb: int = -1
    filter: int = -1
    sp: bool = False

    @property
    def single(self):
        return self.kind in ("frame", "frame16", "frame_rgb", "convert_pad")


PATHS = [Path("planar", "planar"), Path("planar_repitch", "planar", aligned=False),
         Path("planar_in_place", "planar", aligned=False, knob=(("planar_copy", 0),)),
         Path("sp", "sp", sp=True), Path("sp_split", "sp", aligned=False, sp=True),
         Path("sp_prepass", "sp", knob=(("semiplanar_prepass", 1),), sp=True), Path("host", "host")]
PATHS += [Path(f"{'sp' if sp else 'planar'}16_{d}", "d16", depth=d, sp=sp) for sp in (False, True) for d in (10, 12, 16)]
PATHS += [Path(f"down{f}{'_sp' if sp else ''}", "down", factor=f, sp=sp) for sp in (False, True) for f in downscale.FACTORS]
PATHS += [Path(f"rgb_{rgb.NAMES[f]}", "rgb", rgb=f) for f in rgb.FORMATS]
PATHS += [Path(f"resize_{n}{'_sp' if sp else ''}", "resize", filter=f, sp=sp) for sp in (False, True)
          for f, n in zip(resize.FILTERS, ("box", "bilinear", "bicubic"))]
PATHS += [Path("frame", "frame"), Path("frame16", "frame16", depth=12), Path("frame_rgb", "frame_rgb")]
BY_NAME = {p.name: p for p in PATHS}
CONVERT_PAD = Path("convert_pad", "convert_pad")


# ---- geometry and the launch-shape rules of launch_pipeline ---------------------------------------------------------

def n_mcu(w, h, fmt):
    px = 8 if fmt == 2 else 16
    return -(-w // px) * -(-h // 16)


def n_tiles(w, h, fmt):
    return -(-n_mcu(w, h, fmt) // TILE_MCUS)


def n_units(w, h, fmt):
    return -(-n_mcu(w, h, fmt) * (8 if fmt == 1 else 6) // UNIT_BLOCKS)


def roles(fmt):
    return 4 if fmt == 1 else 3


def tiles_per_cta(sizes, fmt, sms=SMS, forced=0):
    """K2's consecutive tiles per CTA for a batch of frames of these (encoded) sizes"""
    if forced:
        return forced
    t = sum(n_tiles(w, h, fmt) for w, h in sizes) * roles(fmt) // (sms * FDCT_MIN_CTAS * 4)
    return min(max(t, 1), MAX_TILES)


def k4b_width(sizes, fmt, sms=SMS):
    """units per warp of scan_place_kernel: 8 when the batch has fewer K4b groups than two per SM"""
    groups = -(-max(n_units(w, h, fmt) for w, h in sizes) // GROUP_UNITS)
    return 8 if groups * len(sizes) < 2 * sms else 32


# ---- cases ---------------------------------------------------------------------------------------------------------

@dataclass(frozen=True)
class Frame:
    w: int           # source size (RGB, 16-bit, downscaled, resized: the caller's frame)
    h: int
    kind: str
    amp: int
    layout: str = "tight"  # device / host placement: tight | pitched (aligned) | shift (base 3 bytes off) | luma16 (chroma pitch odd)
    out: Tuple[int, int] = None  # resize: the encoded size


@dataclass
class Case:
    id: str
    fmt: int
    q: int
    range_mode: int
    path: Path
    form: str
    tiles: int
    k4b: int
    frames: Tuple[Frame, ...]
    rgb_format: int = rgb.RGB24  # frame_rgb
    check: Tuple[int, ...] = field(default=())  # frames whose every stage is compared

    @property
    def settings(self):
        return (self.fmt, self.q, self.range_mode)

    def out_size(self, f: Frame):
        if self.path.kind == "down":
            return -(-f.w // self.path.factor), -(-f.h // self.path.factor)
        return f.out if self.path.kind == "resize" else (f.w, f.h)

    def out_sizes(self):
        return [self.out_size(f) for f in self.frames]

    def params(self):
        return (self.fmt, self.path.name, self.form, self.tiles, self.k4b, (self.q, self.range_mode))


def out_of(path, w, h):
    if path.kind == "down":
        return -(-w // path.factor), -(-h // path.factor)
    return w, h


def valid(fmt, path, form, tiles, k4b, st):
    if path.single or path.kind == "d16":
        if form != "batch":
            return False
        if path.single and k4b == 32:
            return False
    if k4b == 32 and path.kind != "resize":  # the largest frame a source may be, as many of them as a case may have
        return MAX_FRAMES * -(-n_units(*out_of(path, *BIG), fmt) // GROUP_UNITS) >= 2 * SMS
    return True


def pairs(p):
    return {(i, p[i], j, p[j]) for i, j in itertools.combinations(range(len(p)), 2)}


def host_aligned(w, h, fmt):
    """a tight frame at a 256-byte aligned base: every plane's rows on 8-byte boundaries"""
    ch, cw = chroma_shape(w, h, fmt)
    return w % 8 == 0 and cw % 8 == 0 and (w * h) % 8 == 0 and (w * h + cw * ch) % 8 == 0


def realize(params, rng, sms=SMS, rgb_format=None):
    """a Case holding params, its frames drawn by rng"""
    fmt, name, form, tiles, k4b, (q, r) = params
    path = BY_NAME[name]
    small = [s for s in SIZES if s != BIG and min(out_of(path, *s)) >= 2]

    def frame(w, h, big=False):
        kind = "textured" if big or w * h > 1_000_000 else rng.choice(KINDS)
        if path.kind in ("planar", "sp", "d16", "down", "resize"):
            # frames a path reads in place are aligned; a converting path reads any placement
            if path.kind in ("planar", "sp"):
                layout = "pitched" if path.aligned else rng.choice(("shift", "luma16"))
            else:
                layout = rng.choice(("pitched", "tight", "shift", "luma16"))
        else:
            layout = "tight"
        out = None
        if path.kind == "resize":  # a size the filter has to work for: down or up, any ratio, within the encoder's maximum
            out = (3840, 2160) if big else (max(2, int(w * rng.choice((0.37, 0.5, 0.73, 1.0, 1.6)))),
                                            max(2, int(h * rng.choice((0.41, 0.5, 0.8, 1.0, 1.9)))))
            out = (min(out[0], 3840), min(out[1], 4098))
        return Frame(w, h, kind, 10 if big or w * h > 1_000_000 else rng.choice((20, 40, 80)), layout, out)

    if path.single:
        w, h = rng.choice(small)
        frames = [frame(w, h)]
    elif k4b == 8:
        pool = small if path.kind != "down" else small + [BIG]
        if form == "batch":
            w, h = rng.choice(pool)
            f = frame(w, h)
            frames = [f] * rng.randint(1, 3)
        else:
            while True:  # two encoded sizes or more
                frames = [frame(w, h) for w, h in rng.sample(pool, rng.randint(2, 4))]
                if len({out_of(path, f.w, f.h) if f.out is None else f.out for f in frames}) > 1:
                    break
    else:
        src = BIG if path.kind != "resize" else (2562, 1442)
        big = frame(*src, big=True)
        out = out_of(path, *src) if path.kind != "resize" else big.out
        groups = -(-n_units(*out, fmt) // GROUP_UNITS)
        n = -(-2 * sms // groups)
        assert n <= MAX_FRAMES, (params, n)
        if form == "batch":
            frames = [big] * n
        else:
            others = [frame(w, h) for w, h in rng.sample([s for s in small if s[0] * s[1] < 400_000], 2)]
            frames = [big] + [others[i % 2] for i in range(n - 1)]
    case = Case("", fmt, q, r, path, form, tiles, k4b, tuple(frames),
                rgb_format=rgb_format if rgb_format is not None else rng.choice(rgb.FORMATS))
    got = model(case, sms)
    assert got["k4b"] == k4b and got["list"] == (form == "list"), (params, got)
    n = len(frames)
    case.check = tuple(sorted({0, n - 1, rng.randrange(n)}))
    return case


def required():
    """the cases a covering array of pairs would not guarantee: every K2 instantiation with several tiles per CTA on a partial
    last group of tiles, every input kernel in the list form with two sizes or more (16-bit frames have no list call), the
    semi-planar surfaces of a decoder read in place with the automatic tiles per CTA above 1, and h2j_convert_pad"""
    out = []
    for fmt in FMTS:
        for name in ("planar", "sp"):
            for form in FORMS:
                # 2562x1442 (and 641x479) tiles do not divide by 3: the last group of every frame is partial
                frames = (Frame(2562, 1442, "noise", 30, "pitched"), Frame(641, 479, "textured", 40, "pitched"))
                out.append(Case(f"req-k2-{name}-{form}-f{fmt}", fmt, 0, 0, BY_NAME[name], form, 3, 8,
                                frames if form == "list" else frames[:1] * 2))
        # the production case: a list of decoder surfaces read in place, enough of them for the automatic tiles per CTA > 1
        big = Frame(1920, 1080, "textured", 10, "pitched")
        out.append(Case(f"req-sp-list-auto-f{fmt}", fmt, 0, 0, BY_NAME["sp"], "list", 0, 8,
                        (big,) * 12 + (Frame(1918, 1078, "textured", 10, "pitched"),)))
        # unaligned planar frames read in place (as when the slot has no room for their copies): luma rows 16-byte aligned
        # and chroma rows not (K1's vector path, K2's bytewise one), or no row aligned; device and host, both forms
        in_place, host_in_place = BY_NAME["planar_in_place"], Path("host_in_place", "host", knob=(("planar_copy", 0),))
        out.append(Case(f"req-planar-in-place-list-f{fmt}", fmt, 0, 0, in_place, "list", 0, 8,
                        (Frame(1280, 720, "textured", 30, "luma16"), Frame(131, 77, "noise", 60, "shift"))))
        out.append(Case(f"req-planar-in-place-batch-f{fmt}", fmt, 0, 0, in_place, "batch", 0, 8, (Frame(1918, 1078, "textured", 30, "luma16"),) * 3))
        out.append(Case(f"req-host-in-place-batch-f{fmt}", fmt, 0, 0, host_in_place, "batch", 0, 8, (Frame(641, 479, "noise", 20),) * 2))
        out.append(Case(f"req-host-in-place-list-f{fmt}", fmt, 0, 0, host_in_place, "list", 0, 8,
                        (Frame(1918, 1078, "textured", 30), Frame(17, 17, "noise", 60), Frame(33, 47, "blocks", 30))))
    for p in PATHS:
        if p.kind in ("planar", "sp", "host", "down", "rgb", "resize") and not (p.kind in ("planar", "sp") and p.aligned and not p.knob):
            for fmt in ((0, 1, 2) if p.kind == "rgb" else (0,)):
                frames = (Frame(641, 479, "noise", 20, "tight" if p.aligned else "shift", (400, 300)),
                          Frame(33, 47, "blocks", 30, "pitched" if p.aligned else "luma16", (64, 17)))
                out.append(Case(f"req-list-{p.name}-f{fmt}", fmt, 31, 0, p, "list", 0, 8, frames))
    out.append(Case("req-convert_pad", 0, 0, 0, CONVERT_PAD, "batch", 0, 8, (Frame(322, 242, "textured", 40),)))
    for i, c in enumerate(out):
        c.check = tuple(range(len(c.frames))) if len(c.frames) <= 3 else (0, len(c.frames) // 2, len(c.frames) - 1)
    return out


def matrix(sms=SMS):
    """the committed covering array: REQUIRED, then cases chosen greedily (fixed seed) until every valid pair is held"""
    rng = random.Random(SEED)
    space = [p for p in itertools.product(FMTS, [p.name for p in PATHS], FORMS, TILES, K4B, SETTINGS) if valid(p[0], BY_NAME[p[1]], *p[2:])]
    uncovered = set().union(*(pairs(p) for p in space))
    cases = required()
    for c in cases:
        if c.path.name in BY_NAME:
            uncovered -= pairs(c.params())
    by_pair = {}
    for p in space:
        for pr in pairs(p):
            by_pair.setdefault(pr, []).append(p)
    while uncovered:
        first = min(uncovered)
        cands = by_pair[first]
        cands = rng.sample(cands, min(40, len(cands)))
        best = max(cands, key=lambda p: len(pairs(p) & uncovered))
        uncovered -= pairs(best)
        cases.append(realize(best, rng, sms))
    for i, c in enumerate(cases):
        if not c.id:
            fmt, name, form, tiles, k4b, (q, r) = c.params()
            c.id = f"m{i:03d}-{name}-{form}-f{fmt}-t{tiles}-k{k4b}-q{q}r{r}"
    return cases


# ---- the dispatch model ----------------------------------------------------------------------------------------------

def bool_name(x):
    return "true" if x else "false"


def kernel_name(demangled: str) -> str:
    """'void h2j::k<3, true>(h2j::CopyTable, ...)' (c++filt, the profiler) -> 'h2j::k<3, true>'"""
    n = demangled.strip()
    n = n[5:] if n.startswith("void ") else n
    return n.split("(")[0].strip()


def placement(case, f: Frame):
    """(y_pitch, c_pitch, u_off, v_off (None: semi-planar), size, shift) in bytes of a YUV frame as the test places it: rows
    tight, at 64-byte pitches, tight 3 (16-bit: 2) bytes past an aligned base, or luma rows at a 16-byte pitch and chroma
    rows at an odd one (semi-planar: one odd pitch)"""
    p = case.path
    bps = 2 if p.kind == "d16" else 1
    ch, cw = chroma_shape(f.w, f.h, case.fmt)
    yrow, crow = bps * f.w, bps * (2 * cw if p.sp else cw)
    if p.sp:
        yrow = crow = max(yrow, crow)
    yp, cp, shift = yrow, crow, 0
    if f.layout == "pitched":
        yp, cp = align(yrow, 64), align(crow, 64)
    elif f.layout == "shift":
        shift = 3 if bps == 1 else 2
    elif f.layout == "luma16":
        yp, cp = align(yrow, 16), align(crow, 16) + (3 if bps == 1 else 2)
    if p.sp:
        yp = cp = max(yp, cp)
    u_off = yp * f.h
    v_off = None if p.sp else u_off + cp * ch
    return yp, cp, u_off, v_off, (v_off or u_off) + cp * ch, shift


def frame_aligned8(case, f: Frame):
    """the frame's rows all start on 8-byte boundaries where the pipeline would read it in place"""
    if case.path.kind == "host":
        return host_aligned(f.w, f.h, case.fmt)
    yp, cp, u_off, v_off, _, shift = placement(case, f)
    return all(x % 8 == 0 for x in (yp, cp, u_off, v_off or 0, shift))


def model(case: Case, sms=SMS):
    """{'kernels': the demangled names of the kernels the case launches (sorted), 'launches': how many, 'list', 'k4b',
    'tiles_per_cta', 'copy': the input-stage kernel or None}"""
    p, fmt = case.path, case.fmt
    knobs = dict(p.knob)
    if p.kind == "convert_pad":
        return dict(kernels=["h2j::convert_pad_kernel"], launches=1, list=False, k4b=None, tiles_per_cta=None, copy=None)
    sizes = case.out_sizes()
    copy, nv12 = None, False
    if p.kind in ("planar", "host"):
        if knobs.get("planar_copy", 1) and not all(frame_aligned8(case, f) for f in case.frames):
            copy = "h2j::repitch_kernel"
    elif p.kind == "sp":
        if knobs.get("semiplanar_prepass", 0) or not all(frame_aligned8(case, f) for f in case.frames):
            copy = "h2j::nv12_to_i420_kernel"
        else:
            nv12 = True
    elif p.kind in ("d16", "frame16"):
        copy = f"h2j::depth_to_8_kernel<{bool_name(p.sp)}>"
    elif p.kind == "down":
        copy = f"h2j::downscale_list_kernel<{p.factor}, {bool_name(p.sp)}>"
    elif p.kind in ("rgb", "frame_rgb"):
        k = p.rgb if p.kind == "rgb" else case.rgb_format
        copy = f"h2j::rgb_to_planar_kernel<{1 if k == rgb.PLANAR else 4 if k in (rgb.RGBX, rgb.BGRX) else 3}, {fmt}>"
    elif p.kind == "resize":
        copy = f"h2j::resize_list_kernel<{bool_name(p.sp)}>"
    # the batch form: every frame of one layout at one stride.  A case of one encoded size is submitted so that its frames
    # are (one layout at one stride, or copied by the input stage to the slot's buffer at one spacing); two sizes or more
    # make a list
    lst = len(set(sizes)) > 1
    k4b = k4b_width(sizes, fmt, sms)
    tpc = tiles_per_cta(sizes, fmt, sms, case.tiles)
    k2 = f"h2j::fdct_quant_kernel<{bool_name(nv12)}, {bool_name(lst)}>" if fmt == 0 else f"h2j::fdct_quant_fmt_kernel<{fmt}, {bool_name(nv12)}, {bool_name(lst)}>"
    ks = [f"h2j::mbvar_kernel<{bool_name(lst)}>", k2, f"h2j::huffman_kernel<{bool_name(lst)}>", f"h2j::entropy_walk_kernel<{fmt}, {bool_name(lst)}>",
          f"h2j::scan_place_kernel<{k4b}, {bool_name(lst)}>", "h2j::stuff_kernel"]
    if not p.single:
        ks += ["h2j::pack_offsets_kernel", "h2j::pack_kernel"]
    if copy:
        ks.append(copy)
    return dict(kernels=sorted(ks), launches=len(ks), list=lst, k4b=k4b, tiles_per_cta=tpc, copy=copy)


def partial_last_group(case: Case, sms=SMS):
    """some frame's tiles do not fill its last group of tiles_per_cta"""
    t = model(case, sms)["tiles_per_cta"]
    return any(n_tiles(w, h, case.fmt) % t for w, h in case.out_sizes())


def compiled_kernels():
    """the entry functions of the library's build (its ptxas log), demangled by c++filt, without their parameter lists"""
    with open(PTXAS_LOG) as f:
        mangled = sorted(set(re.findall(r"Compiling entry function '(\w+)'", f.read())))
    out = subprocess.run(["c++filt"], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout.split("\n")
    return {kernel_name(n) for n in out if n}


# ---- the expected product of every stage ------------------------------------------------------------------------------

_cache = {}


def source(case: Case, f: Frame):
    """the frame's content before the input stage: (y, u, v) 8-bit planes at the case's chroma format, or for RGB paths the
    (H, W, 3) picture"""
    key = ("src", f.w, f.h, f.kind, f.amp, case.fmt, case.path.kind in ("rgb", "frame_rgb"))
    if key not in _cache:
        from tests.support import oracle as orc

        seed = (f.w * 7919 + f.h * 104729 + KINDS.index(f.kind) * 31) % 100000
        if key[-1]:
            y, u, v = orc.synth_planes_fmt(f.w, f.h, 2, f.kind, seed=seed, amp=f.amp)
            _cache[key] = np.stack([y, u, v], -1)
        else:
            _cache[key] = orc.synth_planes_fmt(f.w, f.h, case.fmt, f.kind, seed=seed, amp=f.amp)
    return _cache[key]


def planes(case: Case, f: Frame):
    """the planar frame the pipeline encodes"""
    p = case.path
    key = ("planes", f, case.fmt, p.kind, p.factor, p.filter, p.rgb, case.rgb_format if p.kind == "frame_rgb" else None)
    if key not in _cache:
        src = source(case, f)
        if p.kind == "down":
            out = downscale.downscale_planar(*src, p.factor)
        elif p.kind == "resize":
            out = resize.resize_planar(*src, *f.out, case.fmt, p.filter)
        elif p.kind in ("rgb", "frame_rgb"):
            k = p.rgb if p.kind == "rgb" else case.rgb_format
            out = rgb.to_planar(rgb.as_format(src, k), k, case.fmt)
        else:
            out = src
        _cache[key] = out
    return _cache[key]


@dataclass
class Expected:
    planes: tuple
    mb_var_sum: int
    qscale: int
    coefs: np.ndarray
    hist: list
    bits: list
    vals: list
    nvals: list
    header_bytes: int
    scan_bits: int
    stuffed_ff: int
    jpeg: bytes


def expected(case: Case, f: Frame) -> Expected:
    """every stage's product for frame f of the case: input planes from the numpy models, K1 .. K4 from the CPU oracle, K5's
    0xFF count from an independent entropy decode of the oracle's JPEG"""
    from tests.support import oracle as orc

    rm = 0 if case.path.kind in ("rgb", "frame_rgb") else case.range_mode  # RGB frames are full range by construction
    pl = planes(case, f)
    key = ("oracle", id(pl), case.fmt, case.q, rm)
    if key not in _cache:
        jpeg, d, coefs = orc.oracle_encode(*pl, fixed_qscale=case.q, range_mode=rm, want_coefs=True, chroma_format=case.fmt)
        _, info = orc.decode_coefs(jpeg)
        _cache[key] = (Expected(pl, d.mb_var_sum, d.qscale, coefs, [list(d.hist[t]) for t in range(4)], [bytes(d.bits[t]) for t in range(4)],
                                [bytes(d.vals[t])[: d.nvals[t]] for t in range(4)], list(d.nvals), d.header_bytes, d.scan_bits, int(info[2]), jpeg), pl)
    return _cache[key][0]


def clear_cache():
    _cache.clear()
