"""GPU: the dispatch matrix (tests/support/dispatch.py), every case against the model stage by stage.

Cases are grouped by encoder settings; each group runs on one long-lived encoder of two slots, the slots alternating, so
that every case also meets the state an earlier batch left in its slot: large frames before small ones, batch form before
list form, converting inputs before frames read in place, the resize arena growing mid-group.  Each case is submitted and
collected before the next one starts.  Every frame's JPEG is compared with the oracle's; for the case's checked frames
(first, last and one seeded) every stage is compared in pipeline order, and a failure names the first stage that diverges.
A mismatch is replayed once on a fresh encoder to tell a slot-history bug from a stateless one; a CUDA error stops the
run.  The launch count of every case is the model's; each group runs under torch.profiler and every h2j kernel it observes
is in the union of its cases' model sets (per group, not per case: profiling every case separately costs more than the
cases); across the groups every kernel the library compiles is observed."""
import numpy as np
import pytest

from tests.support import dispatch as D
from tests.support import rgb as R
from tests.support.layouts import BIG_JPEG, Frames, align, place

pytestmark = pytest.mark.gpu

CASES = D.matrix()
GROUPS = {}
for _c in CASES:
    GROUPS.setdefault(_c.settings, []).append(_c)
OBSERVED = set()
RAN = set()
STOPPED = []


def ordered(cases):
    def key(c):
        m = D.model(c)
        px = max(w * h for w, h in c.out_sizes())
        return (m["list"], m["copy"] is None, px if c.path.kind == "resize" else -px)

    return sorted(cases, key=key)


def widen(p, d, rng):
    """8-bit plane -> 16-bit words holding p in bits [d - 8, d), random bits below and (d < 16) random garbage above"""
    w = (p.astype(np.uint16) << (d - 8)) | rng.integers(0, 1 << (d - 8), p.shape, dtype=np.uint16)
    if d < 16:
        w |= rng.integers(0, 1 << (16 - d), p.shape, dtype=np.uint16) << d
    return w


def yuv_source(case, f):
    y, u, v = D.source(case, f)
    if case.path.depth > 8:
        rng = np.random.default_rng(f.w * 131 + f.h)
        return tuple(widen(x, case.path.depth, rng) for x in (y, u, v))
    return y, u, v


def yuv_bytes(case, f):
    """the frame's bytes as placed (dispatch.placement) and the shift of its base"""
    yp, cp, u_off, v_off, size, shift = D.placement(case, f)
    return place(*yuv_source(case, f), yp, cp, u_off, v_off, size=size), shift


def submit(e, case, slot, keep):
    """enqueue the case; returns None, or the JPEG of a single-picture call"""
    import torch

    import h2j_b200 as H

    p, fr = case.path, Frames()
    keep.append(fr)
    f0, n = case.frames[0], len(case.frames)
    if p.kind == "frame":
        return e.yuv2jpeg(*D.source(case, f0))
    if p.kind == "frame16":
        return e.yuv2jpeg16(*yuv_source(case, f0), p.depth)
    if p.kind == "frame_rgb":
        return e.rgb2jpeg(R.as_format(D.source(case, f0), case.rgb_format), case.rgb_format)
    if p.kind == "host":
        tights = [np.concatenate([x.ravel() for x in D.source(case, f)]) for f in case.frames]
        keep.extend(tights)
        if case.form == "batch":
            arr = np.stack(tights)
            keep.append(arr)
            e.submit_host(slot, arr.ctypes.data, arr.shape[1], n, f0.w, f0.h)
        else:
            e.submit_host_list(slot, [t.ctypes.data for t in tights], [(f.w, f.h) for f in case.frames])
        return None
    if case.form == "batch" and p.kind in ("planar", "sp", "d16"):
        buf, shift = yuv_bytes(case, f0)
        stride = align(buf.size + shift, 256)
        one = np.full(stride, 0xA5, np.uint8)
        one[shift: shift + buf.size] = buf
        d = torch.from_numpy(one).cuda().repeat(n)
        torch.cuda.synchronize()  # the slot runs on its own stream
        keep.append(d)
        yp, cp, u_off, v_off, _, _ = D.placement(case, f0)
        base = d.data_ptr() + shift
        if p.kind == "d16" and p.sp:
            e.submit_device_semiplanar16(slot, base, stride, yp, u_off, p.depth, n, f0.w, f0.h)
        elif p.kind == "d16":
            e.submit_device_pitched16(slot, base, stride, yp, cp, u_off, v_off, p.depth, n, f0.w, f0.h)
        elif p.sp:
            e.submit_device_semiplanar(slot, base, stride, yp, u_off, n, f0.w, f0.h)
        else:
            e.submit_device_pitched(slot, base, stride, yp, cp, u_off, v_off, n, f0.w, f0.h)
        return None
    descs = {}  # frames repeated in a case share their allocation
    for f in case.frames:
        if f in descs:
            continue
        if p.kind == "rgb":
            descs[f] = R.place_rgb(fr, R.as_format(D.source(case, f), p.rgb), p.rgb)
            continue
        buf, shift = yuv_bytes(case, f)
        yp, cp, u_off, v_off, _, _ = D.placement(case, f)
        descs[f] = H.FrameDesc(fr.put(buf, shift), f.w, f.h, yp, cp, u_off, v_off or 0)
    ds = [descs[f] for f in case.frames]
    layout = H.LAYOUT_SEMIPLANAR if p.sp else H.LAYOUT_PLANAR
    if p.kind == "rgb":
        e.submit_device_rgb(slot, p.rgb, ds)
    elif p.kind == "down":
        e.submit_device_downscaled(slot, layout, ds, p.factor)
    elif p.kind == "resize":
        e.submit_device_resized(slot, layout, ds, [f.out for f in case.frames], p.filter)
    else:
        e.submit_device_list(slot, layout, ds)
    return None


def first_divergence(e, slot, case, i, want):
    """None, or (stage, detail) of the first stage of frame i whose product differs from the model's"""
    w, h = case.out_size(case.frames[i])
    got = e.frame_planes(slot, i, w, h)
    for name, g, x in zip("yuv", got, want.planes):
        if g.shape != x.shape or (g != x).any():
            at = np.argwhere(g != x)[0] if g.shape == x.shape else g.shape
            return "input planes", f"plane {name} differs first at {tuple(at)}"
    info = e.frame_info(slot, i)
    if (info.mb_var_sum, info.qscale) != (want.mb_var_sum, want.qscale):
        return "K1", f"mb_var_sum / qscale {info.mb_var_sum} / {info.qscale}, want {want.mb_var_sum} / {want.qscale}"
    coefs = e.coefficients(slot, i, want.coefs.shape[0])
    bad = np.nonzero((coefs != want.coefs).any(axis=1))[0]
    if bad.size:
        return "K2", f"{bad.size} blocks' coefficients differ, first block {bad[0]}"
    for t in range(4):
        if list(info.hist[t]) != want.hist[t]:
            return "K2", f"histogram {t}"
    for t in range(4):
        if info.nvals[t] != want.nvals[t] or bytes(info.bits[t]) != want.bits[t] or bytes(info.vals[t])[: info.nvals[t]] != want.vals[t]:
            return "K3", f"Huffman table {t} (BITS / HUFFVAL)"
    if info.header_bytes != want.header_bytes:
        return "K3", f"header bytes {info.header_bytes}, want {want.header_bytes}"
    if info.scan_bits != want.scan_bits:
        return "K4a/K4b", f"scan bits {info.scan_bits}, want {want.scan_bits}"
    if info.stuffed_ff != want.stuffed_ff:
        return "K5", f"stuffed 0xFF {info.stuffed_ff}, want {want.stuffed_ff}"
    return None


def run_case(e, case, slot, sms):
    """submit and collect the case, then compare; None or a description of the first mismatch"""
    m = D.model(case, sms)
    keep = []
    before = e.kernel_launches
    if case.path.kind == "convert_pad":
        y, u, v = D.source(case, case.frames[0])
        got = e.convert_pad(y, u, v, 0)
        mw, mh = (y.shape[1] + 15) // 16, (y.shape[0] + 15) // 16
        pad = [np.pad(y, ((0, mh * 16 - y.shape[0]), (0, mw * 16 - y.shape[1])), mode="edge")]
        pad += [np.pad(c[: y.shape[0] >> 1, : y.shape[1] >> 1], ((0, mh * 8 - (y.shape[0] >> 1)), (0, mw * 8 - (y.shape[1] >> 1))), mode="edge")
                for c in (u, v)]
        if e.kernel_launches - before != m["launches"]:
            return f"{e.kernel_launches - before} kernel launches, the model says {m['launches']}"
        return "frame 0: first diverging stage input planes (padded)" if any((g != x).any() for g, x in zip(got, pad)) else None
    single = submit(e, case, slot, keep)
    if single is not None:
        jpegs = [single]
    else:
        r = e.collect(slot, strict=False)
        if r.status != [0] * len(case.frames):
            return f"frame status {r.status}"
        jpegs = r.jpegs
    launches = e.kernel_launches - before
    if launches != m["launches"]:
        return f"{launches} kernel launches, the model says {m['launches']}"
    for i, f in enumerate(case.frames):
        want = D.expected(case, f)
        stage = first_divergence(e, 0 if case.path.single else slot, case, i, want) if i in case.check else None
        if stage is None and jpegs[i] != want.jpeg:
            stage = ("JPEG", f"{len(jpegs[i])} bytes, want {len(want.jpeg)}")
        if stage:
            return f"frame {i}: first diverging stage {stage[0]}: {stage[1]}"
    return None


def attempt(e, case, slot, sms):
    """run_case with the case's knobs set; an error the library reports is a mismatch, a CUDA error stops the matrix"""
    import h2j_b200 as H

    for name, value in case.path.knob + (("fdct_tiles_per_cta", case.tiles),):
        e.set_knob(name, value)
    try:
        return run_case(e, case, slot, sms)
    except H.H2JError as x:
        if x.status == H.ERR_CUDA:
            STOPPED.append(f"{case.id}: {x}")
            pytest.fail(f"{case.id}: CUDA error, not rerun: {x}")
        return f"error {x}"
    finally:
        for name, _ in case.path.knob:
            e.set_knob(name, {"planar_copy": 1}.get(name, 0))


def encoder_for(cases, settings):
    import h2j_b200 as H

    fmt, q, rm = settings
    sizes = [s for c in cases for s in c.out_sizes()]
    return H.Encoder(max_width=max(w for w, _ in sizes), max_height=max(h for _, h in sizes), max_batch=max(len(c.frames) for c in cases),
                     n_slots=2, chroma_format=fmt, fixed_qscale=q, range_mode=rm, max_jpeg_bytes=BIG_JPEG)


@pytest.mark.parametrize("settings", sorted(GROUPS), ids=lambda s: f"f{s[0]}-q{s[1]}-r{s[2]}")
def test_group(orc, settings):
    import torch
    from torch.profiler import ProfilerActivity, profile

    if STOPPED:
        pytest.skip(f"a CUDA error stopped the matrix: {STOPPED[0]}")
    RAN.add(settings)
    cases = ordered(GROUPS[settings])
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    failures = []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        torch.ones(1, device="cuda").add_(1)  # the activity trace is live before the group's first kernel
        torch.cuda.synchronize()
        with encoder_for(cases, settings) as e:
            for k, case in enumerate(cases):
                err = attempt(e, case, k % 2, sms)
                if err:
                    with encoder_for([case], settings) as fresh:
                        again = attempt(fresh, case, 0, sms)
                    failures.append(f"{case.id}: {err} ({'stateless' if again else 'depends on slot history'})")
        torch.cuda.synchronize()
    D.clear_cache()
    seen = {D.kernel_name(ev.name) for ev in prof.events()}
    seen = {n for n in seen if n.startswith("h2j::")}
    OBSERVED.update(seen)
    want = set().union(*(D.model(c, sms)["kernels"] for c in cases))
    assert not failures, "\n".join(failures)
    # the activity trace may drop a record, so a kernel missing here is not a finding by itself (the launch counts are
    # exact, and test_every_compiled_kernel_was_observed needs each kernel seen in some group); one outside the model is
    assert seen <= want, f"profiled kernels beyond the model's: {sorted(seen - want)}"


def test_every_compiled_kernel_was_observed():
    if RAN != set(GROUPS):
        pytest.skip(f"{len(RAN)} of {len(GROUPS)} groups ran")
    want = D.compiled_kernels()
    assert OBSERVED == want, f"never observed: {sorted(want - OBSERVED)}; unknown: {sorted(OBSERVED - want)}"
