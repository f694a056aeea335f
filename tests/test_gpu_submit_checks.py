"""GPU suite: the argument checks of every submit entry point, table-driven, on a 4:2:0 and a 4:4:4 encoder.  Every
malformed call must return its status and leave the slot as it was: a batch in flight stays collectable with its JPEGs, a
collected batch keeps its frame_info, and the slot takes the next valid batch as if the call had not happened."""
import ctypes as C

import numpy as np
import pytest

from tests.support.layouts import align

pytestmark = pytest.mark.gpu

W, H, B = 64, 32, 2  # the encoder's maximum and batch


class Dims:
    """the byte sizes every call of the table is made of, at one chroma format"""

    def __init__(self, fmt):
        import h2j_b200

        self.fmt = fmt
        self.ch, self.cw = h2j_b200.chroma_shape(W, H, fmt)
        self.pairs = 2 * self.cw  # a row of Cb/Cr pairs: as long as a luma row at 4:2:0, twice as long at 4:4:4
        self.sp = max(W, self.pairs)  # the pitch of a tight semi-planar frame
        self.tight = W * H + 2 * self.cw * self.ch  # a tight planar frame
        self.sp_size = self.sp * (H + self.ch)  # a tight semi-planar frame
        self.stride = align(max(self.tight, self.sp_size), 4096)  # holds either (16-bit frames: twice this)


def _lib():
    import h2j_b200

    return h2j_b200.load_library()


def _tight(w, h, fmt):
    """(y_pitch, c_pitch, u_offset, v_offset) of a w x h planar frame packed tight"""
    import h2j_b200

    ch, cw = h2j_b200.chroma_shape(w, h, fmt)
    return w, cw, w * h, w * h + cw * ch


def _descs(ptrs, w, h, y_pitch, c_pitch, u_off, v_off):
    import h2j_b200

    return (h2j_b200.FrameDesc * len(ptrs))(*[h2j_b200.FrameDesc(p, w, h, y_pitch, c_pitch, u_off, v_off) for p in ptrs])


class Env:
    """device and host memory holding valid frames for every entry point"""

    def __init__(self):
        import torch

        rng = np.random.default_rng(11)
        self.host = rng.integers(0, 256, 1 << 20, dtype=np.uint8)
        self.host16 = rng.integers(0, 1024, 1 << 16, dtype=np.uint16)
        self.dev = torch.from_numpy(self.host).cuda()
        torch.cuda.synchronize()  # the slot runs on its own stream
        self.p = self.dev.data_ptr()
        self.hp = self.host.ctypes.data


def _planes(arrs, offsets=(0, 0, 0)):
    return (C.c_void_p * 3)(*[a.ctypes.data + o for a, o in zip(arrs, offsets)])


def _strides(s):
    return (C.c_int * 3)(*s)


def submits(e, env, g):
    """entry point -> call(slot=0, **overrides) returning the status; the defaults describe a valid batch of B frames"""
    import h2j_b200

    L, h = _lib(), e._h
    p, hp, S = env.p, env.hp, g.stride
    out = np.empty(1 << 20, np.uint8)
    size = C.c_size_t(0)
    y8, c8 = env.host[: W * H].reshape(H, W), env.host[W * H: W * H + g.cw * g.ch].reshape(g.ch, g.cw)
    y16, c16 = env.host16[: W * H].reshape(H, W), env.host16[W * H: W * H + g.cw * g.ch].reshape(g.ch, g.cw)

    def list_call(fn, layout=h2j_b200.LAYOUT_PLANAR, n=B, frames="ok", null_frame=False, w=W, hh=H, **kw):
        a = dict(zip(("y_pitch", "c_pitch", "u_off", "v_off"), _tight(w, hh, g.fmt)), data=p)
        a.update(kw)
        ptrs = [a["data"] + (i * S if a["data"] else 0) for i in range(B)]
        if null_frame:
            ptrs[1] = 0
        d = _descs(ptrs, w, hh, a["y_pitch"], a["c_pitch"], a["u_off"], a["v_off"])
        return fn(h, a.get("slot", 0), layout, None if frames is None else d, n, *a.get("extra", ()))

    def host_list(n=B, frames="ok", widths="ok", null_frame=False, w=W, hh=H, slot=0):
        ptrs = (C.c_void_p * B)(*[hp + i * S for i in range(B)])
        if null_frame:
            ptrs[1] = None
        ws, hs = (C.c_int * B)(*[w] * B), (C.c_int * B)(*[hh] * B)
        return L.h2j_submit_host_list(h, slot, None if frames is None else ptrs, None if widths is None else ws, hs, n)

    yp, cp, uo, vo = _tight(W, H, g.fmt)
    calls = {
        "device": lambda slot=0, ptr=p, stride=S, n=B, w=W, hh=H: L.h2j_submit_device(h, slot, ptr, stride, n, w, hh),
        "host": lambda slot=0, ptr=hp, stride=S, n=B, w=W, hh=H: L.h2j_submit_host(h, slot, ptr, stride, n, w, hh),
        "semiplanar": lambda slot=0, ptr=p, stride=S, pitch=g.sp, uv=g.sp * H, n=B, w=W, hh=H:
            L.h2j_submit_device_semiplanar(h, slot, ptr, stride, pitch, uv, n, w, hh),
        "nv12": lambda slot=0, ptr=p, stride=S, pitch=g.sp, uv=g.sp * H, n=B, w=W, hh=H:
            L.h2j_submit_device_nv12(h, slot, ptr, stride, pitch, uv, n, w, hh),
        "pitched": lambda slot=0, ptr=p, stride=S, yp=yp, cp=cp, uo=uo, vo=vo, n=B, w=W, hh=H:
            L.h2j_submit_device_pitched(h, slot, ptr, stride, yp, cp, uo, vo, n, w, hh),
        "semiplanar16": lambda slot=0, ptr=p, stride=2 * S, pitch=2 * g.sp, uv=2 * g.sp * H, bd=10, n=B, w=W, hh=H:
            L.h2j_submit_device_semiplanar16(h, slot, ptr, stride, pitch, uv, bd, n, w, hh),
        "pitched16": lambda slot=0, ptr=p, stride=2 * S, yp=2 * yp, cp=2 * cp, uo=2 * uo, vo=2 * vo, bd=10, n=B, w=W, hh=H:
            L.h2j_submit_device_pitched16(h, slot, ptr, stride, yp, cp, uo, vo, bd, n, w, hh),
        "device_list": lambda **kw: list_call(L.h2j_submit_device_list, **kw),
        "downscaled": lambda factor=2, w=2 * W, hh=2 * H, **kw: list_call(L.h2j_submit_device_downscaled, w=w, hh=hh, extra=(factor,), **kw),
        "host_list": host_list,
        "encode_frame": lambda planes="ok", strides=(W, g.cw, g.cw), w=W, hh=H: L.h2j_encode_frame(
            h, None if planes is None else _planes((y8, c8, c8)), _strides(strides), w, hh, out.ctypes.data, out.size, C.byref(size)),
        "encode_frame16": lambda planes="ok", offsets=(0, 0, 0), strides=(2 * W, 2 * g.cw, 2 * g.cw), bd=10, w=W, hh=H: L.h2j_encode_frame16(
            h, None if planes is None else _planes((y16, c16, c16), offsets), _strides(strides), bd, w, hh, out.ctypes.data, out.size,
            C.byref(size)),
    }
    if g.fmt != h2j_b200.CHROMA_420:
        del calls["nv12"]  # refused whatever its arguments (test_nv12_refuses_other_chroma_formats)
    return calls


def malformed_cases(g):
    """(entry point, what is wrong, overrides, expected status)"""
    import h2j_b200

    INV, UNS = h2j_b200.ERR_INVALID_ARG, h2j_b200.ERR_UNSUPPORTED
    cw, ch, S = g.cw, g.ch, g.stride
    big = 4 * S  # strides that hold a frame twice the maximum width
    semiplanar8 = ["semiplanar", "nv12"] if g.fmt == h2j_b200.CHROMA_420 else ["semiplanar"]
    cases = []
    for name in ["device", "host", "pitched", "semiplanar16", "pitched16"] + semiplanar8:
        cases += [
            (name, "slot -1", dict(slot=-1), INV),
            (name, "slot past n_slots", dict(slot=2), INV),
            (name, "null pointer", dict(ptr=0), INV),
            (name, "n 0", dict(n=0), INV),
            (name, "n past max_batch", dict(n=B + 1), INV),
            (name, "1 sample wide", dict(w=1), UNS),
        ]
    cases += [
        ("device", "plane past frame_stride", dict(stride=g.tight - 1), INV),
        ("device", "wider than the maximum", dict(w=2 * W, stride=big), UNS),
        ("host", "plane past frame_stride", dict(stride=g.tight - 1), INV),
        ("host", "wider than the maximum", dict(w=2 * W, stride=big), UNS),
    ]
    for name in semiplanar8:
        cases += [
            (name, "pitch shorter than a luma row", dict(pitch=W - 1), INV),
            (name, "pitch shorter than a row of pairs", dict(pitch=g.pairs - 1), INV),
            (name, "pair plane inside the luma plane", dict(uv=g.sp * H - 1), INV),
            (name, "pair plane past frame_stride", dict(stride=g.sp_size - 1), INV),
            (name, "wider than the maximum", dict(w=2 * W, pitch=2 * g.sp, uv=2 * g.sp * H, stride=big), UNS),
            (name, "taller than the maximum", dict(hh=2 * H, uv=2 * g.sp * H, stride=big), UNS),
        ]
    cases += [
        ("pitched", "short luma pitch", dict(yp=W - 1), INV),
        ("pitched", "short chroma pitch", dict(cp=cw - 1), INV),
        ("pitched", "luma plane past frame_stride", dict(stride=W * H - 1, uo=0, vo=0), INV),
        ("pitched", "Cb plane past frame_stride", dict(uo=S - cw * ch + 1), INV),
        ("pitched", "Cr plane past frame_stride", dict(vo=S - cw * ch + 1), INV),
        ("pitched", "wider than the maximum", dict(w=2 * W, yp=2 * W, cp=2 * cw, uo=2 * W * H, vo=2 * (W * H + cw * ch), stride=big), UNS),
    ]
    for name in ("semiplanar16", "pitched16"):
        cases += [
            (name, "bit_depth 8", dict(bd=8), INV),
            (name, "bit_depth 17", dict(bd=17), INV),
            (name, "odd pointer", dict(ptr=1 << 20), INV),  # replaced by an odd device address below
            (name, "odd frame_stride", dict(stride=2 * S - 1), INV),
        ]
    cases += [
        ("semiplanar16", "odd pitch", dict(pitch=2 * g.sp + 1), INV),
        ("semiplanar16", "odd uv_offset", dict(uv=2 * g.sp * H + 1), INV),
        ("semiplanar16", "pitch shorter than a luma row", dict(pitch=2 * W - 2), INV),
        ("semiplanar16", "pitch shorter than a row of pairs", dict(pitch=2 * g.pairs - 2), INV),
        ("semiplanar16", "pair plane inside the luma plane", dict(uv=2 * g.sp * H - 2), INV),
        ("semiplanar16", "pair plane past frame_stride", dict(stride=2 * g.sp_size - 2), INV),
        ("semiplanar16", "wider than the maximum", dict(w=2 * W, pitch=4 * g.sp, uv=4 * g.sp * H, stride=2 * big), UNS),
        ("pitched16", "odd luma pitch", dict(yp=2 * W + 1), INV),
        ("pitched16", "odd chroma pitch", dict(cp=2 * cw + 1), INV),
        ("pitched16", "odd u_offset", dict(uo=2 * W * H + 1), INV),
        ("pitched16", "odd v_offset", dict(vo=2 * (W * H + cw * ch) + 1), INV),
        ("pitched16", "short luma pitch", dict(yp=2 * W - 2), INV),
        ("pitched16", "short chroma pitch", dict(cp=2 * cw - 2), INV),
        ("pitched16", "luma plane past frame_stride", dict(stride=2 * W * H - 2, uo=0, vo=0), INV),
        ("pitched16", "Cb plane past frame_stride", dict(uo=2 * S - 2 * cw * ch + 2), INV),
        ("pitched16", "Cr plane past frame_stride", dict(vo=2 * S - 2 * cw * ch + 2), INV),
        ("pitched16", "wider than the maximum", dict(w=2 * W, yp=4 * W, cp=4 * cw, uo=4 * W * H, vo=4 * (W * H + cw * ch), stride=2 * big), UNS),
    ]
    for name in ("device_list", "downscaled"):
        cases += [
            (name, "slot past n_slots", dict(slot=2), INV),
            (name, "null frames", dict(frames=None), INV),
            (name, "n 0", dict(n=0), INV),
            (name, "n past max_batch", dict(n=B + 1), INV),
            (name, "bad layout", dict(layout=2), INV),
            (name, "null frame data", dict(data=0), INV),
            (name, "null data in the second frame only", dict(null_frame=True), INV),
        ]
    cases += [
        ("device_list", "short luma pitch", dict(y_pitch=W - 1), INV),
        ("device_list", "short chroma pitch", dict(c_pitch=cw - 1), INV),
        ("device_list", "short semi-planar pitch", dict(layout=1, c_pitch=g.pairs - 1, u_off=W * H), INV),
        ("device_list", "pair plane inside the luma plane", dict(layout=1, c_pitch=g.pairs, u_off=W * H - 1), INV),
        ("device_list", "1 sample wide", dict(w=1), UNS),
        ("device_list", "wider than the maximum", dict(w=2 * W), UNS),
        ("device_list", "taller than the maximum", dict(hh=2 * H), UNS),
        ("device_list", "wider than 65500 samples", dict(w=70000), UNS),
        ("downscaled", "factor 3", dict(factor=3), INV),
        ("downscaled", "factor 1", dict(factor=1), INV),
        ("downscaled", "short luma pitch", dict(y_pitch=2 * W - 1), INV),
        ("downscaled", "pair plane inside the luma plane", dict(layout=1, c_pitch=2 * g.pairs, u_off=4 * W * H - 1), INV),
        ("downscaled", "downscaled wider than the maximum", dict(w=4 * W), UNS),
        ("downscaled", "downscaled taller than the maximum", dict(hh=4 * H), UNS),
        ("downscaled", "downscaled smaller than 2x2", dict(w=2, hh=2), UNS),
        ("host_list", "slot past n_slots", dict(slot=2), INV),
        ("host_list", "null frames", dict(frames=None), INV),
        ("host_list", "null sizes", dict(widths=None), INV),
        ("host_list", "n 0", dict(n=0), INV),
        ("host_list", "n past max_batch", dict(n=B + 1), INV),
        ("host_list", "null frame pointer", dict(null_frame=True), INV),
        ("host_list", "1 sample wide", dict(w=1), UNS),
        ("host_list", "wider than the maximum", dict(w=2 * W), UNS),
        ("host_list", "taller than the maximum", dict(hh=2 * H), UNS),
        ("encode_frame", "null planes", dict(planes=None), INV),
        ("encode_frame", "short luma stride", dict(strides=(W - 1, cw, cw)), INV),
        ("encode_frame", "short chroma stride", dict(strides=(W, cw - 1, cw)), INV),
        ("encode_frame", "wider than the maximum", dict(w=2 * W, strides=(2 * W, 2 * cw, 2 * cw)), UNS),
        ("encode_frame16", "null planes", dict(planes=None), INV),
        ("encode_frame16", "bit_depth 8", dict(bd=8), INV),
        ("encode_frame16", "bit_depth 17", dict(bd=17), INV),
        ("encode_frame16", "odd plane pointer", dict(offsets=(1, 0, 0)), INV),
        ("encode_frame16", "odd stride", dict(strides=(2 * W + 1, 2 * cw, 2 * cw)), INV),
        ("encode_frame16", "short luma stride", dict(strides=(2 * W - 2, 2 * cw, 2 * cw)), INV),
        ("encode_frame16", "short chroma stride", dict(strides=(2 * W, 2 * cw - 2, 2 * cw)), INV),
        ("encode_frame16", "wider than the maximum", dict(w=2 * W, strides=(4 * W, 4 * cw, 4 * cw)), UNS),
    ]
    return cases


def _info_bytes(e, slot, frame):
    info = e.frame_info(slot, frame)
    return C.string_at(C.addressof(info), C.sizeof(info))


def test_malformed_submits_leave_the_slot_as_it_was():
    _check_the_table(0)


def test_malformed_submits_at_444_leave_the_slot_as_it_was():
    """4:4:4: a row of pairs is twice a luma row, and chroma rows are as long as luma rows"""
    _check_the_table(2)


def _check_the_table(fmt):
    import h2j_b200

    env = Env()
    g = Dims(fmt)
    with h2j_b200.Encoder(max_width=W, max_height=H, max_batch=B, n_slots=2, chroma_format=fmt) as e:
        calls = submits(e, env, g)
        # the previous batch: a list of two frames of different sizes, so that frame_info differs per frame
        prev = _descs([env.p, env.p + g.stride], W, H, *_tight(W, H, fmt))
        prev[1].width, prev[1].height = 48, 16
        prev[1].y_pitch, prev[1].c_pitch, prev[1].u_offset, prev[1].v_offset = _tight(48, 16, fmt)

        def submit_prev():
            e.submit_device_list(0, h2j_b200.LAYOUT_PLANAR, list(prev))

        submit_prev()
        want = e.collect(0)
        assert want.status == [0, 0]
        infos = [_info_bytes(e, 0, i) for i in range(2)]

        # a batch in flight: every entry point refuses a valid call on its slot, and the batch stays collectable
        submit_prev()
        for name, call in calls.items():
            assert call() == h2j_b200.ERR_BUSY, f"{name}: a valid call on a busy slot"
        got = e.collect(0)
        assert got.jpegs == want.jpegs and got.status == want.status
        assert [_info_bytes(e, 0, i) for i in range(2)] == infos

        # every malformed call on the idle slot returns its status and changes nothing
        wrong = []
        for name, what, kw, status in malformed_cases(g):
            if what == "odd pointer":
                kw = dict(kw, ptr=env.p + 1)
            rc = calls[name](**kw)
            if rc != status:
                wrong.append(f"{name}, {what}: status {rc}, expected {status}")
            if rc == 0 and name not in ("encode_frame", "encode_frame16"):
                e.collect(0 if kw.get("slot", 0) in (0, -1) else kw["slot"], strict=False)
        assert not wrong, "\n".join(wrong)
        assert [_info_bytes(e, 0, i) for i in range(2)] == infos, "a rejected call changed the last batch's frame_info"
        with pytest.raises(h2j_b200.H2JError) as ei:
            e.collect(0)  # nothing in flight: no rejected call left the slot busy
        assert ei.value.status == h2j_b200.ERR_BUSY
        submit_prev()
        got = e.collect(0)
        assert got.jpegs == want.jpegs and got.status == want.status
        assert [_info_bytes(e, 0, i) for i in range(2)] == infos

        # and the valid calls the table starts from are accepted
        for name, call in calls.items():
            assert call() == 0, f"{name}: the valid call was refused: {e._lib.h2j_last_error(e._h)}"
            if name not in ("encode_frame", "encode_frame16"):
                assert e.collect(0).status == [0] * B, name


def test_nv12_refuses_other_chroma_formats():
    import h2j_b200

    env = Env()
    for fmt in (h2j_b200.CHROMA_422, h2j_b200.CHROMA_444):
        with h2j_b200.Encoder(max_width=W, max_height=H, max_batch=B, n_slots=1, chroma_format=fmt) as e:
            assert e._lib.h2j_submit_device_nv12(e._h, 0, env.p, 8192, 2 * W, 2 * W * H, B, W, H) == h2j_b200.ERR_UNSUPPORTED
