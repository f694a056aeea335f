"""GPU suite: the argument checks of every submit entry point, table-driven.  Every malformed call must return its status and
leave the slot as it was: a batch in flight stays collectable with its JPEGs, a collected batch keeps its frame_info, and
the slot takes the next valid batch as if the call had not happened."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W, H, B = 64, 32, 2  # the encoder's maximum (4:2:0) and batch
TIGHT = W * H + 2 * (W // 2) * (H // 2)  # 3072
STRIDE = 4096


def _lib():
    import h2j_b200

    return h2j_b200.load_library()


def _descs(ptrs, w, h, y_pitch, c_pitch, u_off, v_off):
    import h2j_b200

    return (h2j_b200.FrameDesc * len(ptrs))(*[h2j_b200.FrameDesc(p, w, h, y_pitch, c_pitch, u_off, v_off) for p in ptrs])


class Env:
    """device and host memory holding valid frames for every entry point"""

    def __init__(self):
        import torch

        rng = np.random.default_rng(11)
        self.host = rng.integers(0, 256, 1 << 20, dtype=np.uint8)
        self.dev = torch.from_numpy(self.host).cuda()
        torch.cuda.synchronize()  # the slot runs on its own stream
        self.p = self.dev.data_ptr()
        self.hp = self.host.ctypes.data
        self.planes16 = [np.ascontiguousarray(rng.integers(0, 1024, (h, w), dtype=np.uint16)) for (h, w) in ((H, W), (H // 2, W // 2), (H // 2, W // 2))]


def _planes(arrs, offsets=(0, 0, 0)):
    return (C.c_void_p * 3)(*[a.ctypes.data + o for a, o in zip(arrs, offsets)])


def _strides(s):
    return (C.c_int * 3)(*s)


def submits(e, env):
    """entry point -> call(slot=0, **overrides) returning the status; the defaults describe a valid batch of B frames"""
    L, h = _lib(), e._h
    p, hp = env.p, env.hp
    out = np.empty(1 << 20, np.uint8)
    size = C.c_size_t(0)
    y8 = env.host[: W * H].reshape(H, W)
    c8 = env.host[W * H: W * H + (W // 2) * (H // 2)].reshape(H // 2, W // 2)
    import h2j_b200

    def list_call(fn, layout=h2j_b200.LAYOUT_PLANAR, n=B, frames="ok", w=W, h_=H, **kw):
        a = dict(w=w, h=h_, y_pitch=w, c_pitch=w // 2, u_off=w * h_, v_off=w * h_ + (w // 2) * (h_ // 2), data=p)
        a.update(kw)
        ptrs = [a["data"] + (i * STRIDE if a["data"] else 0) for i in range(B)]
        d = _descs(ptrs, a["w"], a["h"], a["y_pitch"], a["c_pitch"], a["u_off"], a["v_off"])
        return fn(h, 0 if "slot" not in a else a["slot"], layout, None if frames is None else d, n, *a.get("extra", ()))

    def host_list(n=B, frames="ok", widths="ok", null_frame=False, w=W, hh=H, slot=0):
        ptrs = (C.c_void_p * B)(*[hp + i * STRIDE for i in range(B)])
        if null_frame:
            ptrs[1] = None
        ws, hs = (C.c_int * B)(*[w] * B), (C.c_int * B)(*[hh] * B)
        return L.h2j_submit_host_list(h, slot, None if frames is None else ptrs, None if widths is None else ws, hs, n)

    return {
        "device": lambda slot=0, ptr=p, stride=STRIDE, n=B, w=W, hh=H: L.h2j_submit_device(h, slot, ptr, stride, n, w, hh),
        "host": lambda slot=0, ptr=hp, stride=STRIDE, n=B, w=W, hh=H: L.h2j_submit_host(h, slot, ptr, stride, n, w, hh),
        "semiplanar": lambda slot=0, ptr=p, stride=STRIDE, pitch=W, uv=W * H, n=B, w=W, hh=H:
            L.h2j_submit_device_semiplanar(h, slot, ptr, stride, pitch, uv, n, w, hh),
        "nv12": lambda slot=0, ptr=p, stride=STRIDE, pitch=W, uv=W * H, n=B, w=W, hh=H:
            L.h2j_submit_device_nv12(h, slot, ptr, stride, pitch, uv, n, w, hh),
        "pitched": lambda slot=0, ptr=p, stride=STRIDE, yp=W, cp=W // 2, uo=2048, vo=2560, n=B, w=W, hh=H:
            L.h2j_submit_device_pitched(h, slot, ptr, stride, yp, cp, uo, vo, n, w, hh),
        "semiplanar16": lambda slot=0, ptr=p, stride=8192, pitch=2 * W, uv=2 * W * H, bd=10, n=B, w=W, hh=H:
            L.h2j_submit_device_semiplanar16(h, slot, ptr, stride, pitch, uv, bd, n, w, hh),
        "pitched16": lambda slot=0, ptr=p, stride=8192, yp=2 * W, cp=W, uo=4096, vo=5120, bd=10, n=B, w=W, hh=H:
            L.h2j_submit_device_pitched16(h, slot, ptr, stride, yp, cp, uo, vo, bd, n, w, hh),
        "device_list": lambda **kw: list_call(L.h2j_submit_device_list, **kw),
        "downscaled": lambda factor=2, w=2 * W, h=2 * H, **kw: list_call(L.h2j_submit_device_downscaled, w=w, h_=h, extra=(factor,), **kw),
        "host_list": host_list,
        "encode_frame": lambda planes="ok", strides=(W, W // 2, W // 2), w=W, hh=H: L.h2j_encode_frame(
            h, None if planes is None else _planes((y8, c8, c8)), _strides(strides), w, hh, out.ctypes.data, out.size, C.byref(size)),
        "encode_frame16": lambda planes="ok", offsets=(0, 0, 0), strides=(2 * W, W, W), bd=10, w=W, hh=H: L.h2j_encode_frame16(
            h, None if planes is None else _planes(env.planes16, offsets), _strides(strides), bd, w, hh, out.ctypes.data, out.size,
            C.byref(size)),
    }


def malformed_cases():
    """(entry point, what is wrong, overrides, expected status)"""
    import h2j_b200

    INV, UNS = h2j_b200.ERR_INVALID_ARG, h2j_b200.ERR_UNSUPPORTED
    cases = []
    batch = ["device", "host", "semiplanar", "nv12", "pitched", "semiplanar16", "pitched16"]
    for name in batch:
        cases += [
            (name, "slot -1", dict(slot=-1), INV),
            (name, "slot past n_slots", dict(slot=2), INV),
            (name, "null pointer", dict(ptr=0), INV),
            (name, "n 0", dict(n=0), INV),
            (name, "n past max_batch", dict(n=B + 1), INV),
            (name, "1 sample wide", dict(w=1), UNS),
        ]
    big = 4 * STRIDE  # strides that hold a frame twice the maximum width
    cases += [
        ("device", "plane past frame_stride", dict(stride=TIGHT - 1), INV),
        ("device", "wider than the maximum", dict(w=2 * W, stride=big), UNS),
        ("host", "plane past frame_stride", dict(stride=TIGHT - 1), INV),
        ("host", "wider than the maximum", dict(w=2 * W, stride=big), UNS),
    ]
    for name in ("semiplanar", "nv12"):
        cases += [
            (name, "short pitch", dict(pitch=W - 1), INV),
            (name, "pair plane inside the luma plane", dict(uv=W * H - 1), INV),
            (name, "pair plane past frame_stride", dict(stride=TIGHT - 1), INV),
            (name, "wider than the maximum", dict(w=2 * W, pitch=2 * W, uv=2 * W * H, stride=big), UNS),
            (name, "taller than the maximum", dict(hh=2 * H, uv=2 * W * H, stride=big), UNS),
        ]
    cases += [
        ("pitched", "short luma pitch", dict(yp=W - 1), INV),
        ("pitched", "short chroma pitch", dict(cp=W // 2 - 1), INV),
        ("pitched", "luma plane past frame_stride", dict(stride=W * H - 1, uo=0, vo=0), INV),
        ("pitched", "Cb plane past frame_stride", dict(uo=STRIDE - 511), INV),
        ("pitched", "Cr plane past frame_stride", dict(vo=STRIDE - 511), INV),
        ("pitched", "wider than the maximum", dict(w=2 * W, yp=2 * W, cp=W, uo=4 * W * H, vo=5 * W * H, stride=big), UNS),
    ]
    for name in ("semiplanar16", "pitched16"):
        cases += [
            (name, "bit_depth 8", dict(bd=8), INV),
            (name, "bit_depth 17", dict(bd=17), INV),
            (name, "odd pointer", dict(ptr=1 << 20), INV),  # replaced by an odd device address below
            (name, "odd frame_stride", dict(stride=8191), INV),
        ]
    cases += [
        ("semiplanar16", "odd pitch", dict(pitch=2 * W + 1), INV),
        ("semiplanar16", "odd uv_offset", dict(uv=2 * W * H + 1), INV),
        ("semiplanar16", "short pitch", dict(pitch=2 * W - 2), INV),
        ("semiplanar16", "pair plane inside the luma plane", dict(uv=2 * W * H - 2), INV),
        ("semiplanar16", "pair plane past frame_stride", dict(stride=6144 - 2), INV),
        ("semiplanar16", "wider than the maximum", dict(w=2 * W, pitch=4 * W, uv=4 * W * H, stride=big), UNS),
        ("pitched16", "odd luma pitch", dict(yp=2 * W + 1), INV),
        ("pitched16", "odd chroma pitch", dict(cp=W + 1), INV),
        ("pitched16", "odd u_offset", dict(uo=4097), INV),
        ("pitched16", "odd v_offset", dict(vo=5121), INV),
        ("pitched16", "short luma pitch", dict(yp=2 * W - 2), INV),
        ("pitched16", "short chroma pitch", dict(cp=W - 2), INV),
        ("pitched16", "luma plane past frame_stride", dict(stride=4096 - 2, uo=0, vo=0), INV),
        ("pitched16", "Cb plane past frame_stride", dict(uo=8192 - 1022), INV),
        ("pitched16", "Cr plane past frame_stride", dict(vo=8192 - 1022), INV),
        ("pitched16", "wider than the maximum", dict(w=2 * W, yp=4 * W, cp=2 * W, uo=8 * W * H, vo=10 * W * H, stride=2 * big), UNS),
    ]
    for name in ("device_list", "downscaled"):
        cases += [
            (name, "slot past n_slots", dict(slot=2), INV),
            (name, "null frames", dict(frames=None), INV),
            (name, "n 0", dict(n=0), INV),
            (name, "n past max_batch", dict(n=B + 1), INV),
            (name, "bad layout", dict(layout=2), INV),
            (name, "null frame data", dict(data=0), INV),
        ]
    cases += [
        ("device_list", "short luma pitch", dict(y_pitch=W - 1), INV),
        ("device_list", "short chroma pitch", dict(c_pitch=W // 2 - 1), INV),
        ("device_list", "short semi-planar pitch", dict(layout=1, c_pitch=W - 1, u_off=W * H), INV),
        ("device_list", "pair plane inside the luma plane", dict(layout=1, c_pitch=W, u_off=W * H - 1), INV),
        ("device_list", "1 sample wide", dict(w=1), UNS),
        ("device_list", "wider than the maximum", dict(w=2 * W, y_pitch=2 * W, c_pitch=W, u_off=2 * W * H, v_off=3 * W * H), UNS),
        ("downscaled", "factor 3", dict(factor=3), INV),
        ("downscaled", "factor 1", dict(factor=1), INV),
        ("downscaled", "short luma pitch", dict(y_pitch=2 * W - 1), INV),
        ("downscaled", "pair plane inside the luma plane", dict(layout=1, c_pitch=2 * W, u_off=4 * W * H - 1), INV),
        ("downscaled", "downscaled wider than the maximum", dict(w=4 * W), UNS),
        ("downscaled", "downscaled smaller than 2x2", dict(w=2, h=2), UNS),
        ("host_list", "slot past n_slots", dict(slot=2), INV),
        ("host_list", "null frames", dict(frames=None), INV),
        ("host_list", "null sizes", dict(widths=None), INV),
        ("host_list", "n 0", dict(n=0), INV),
        ("host_list", "n past max_batch", dict(n=B + 1), INV),
        ("host_list", "null frame pointer", dict(null_frame=True), INV),
        ("host_list", "1 sample wide", dict(w=1), UNS),
        ("host_list", "wider than the maximum", dict(w=2 * W), UNS),
        ("encode_frame", "null planes", dict(planes=None), INV),
        ("encode_frame", "short stride", dict(strides=(W - 1, W // 2, W // 2)), INV),
        ("encode_frame", "wider than the maximum", dict(w=2 * W, strides=(2 * W, W, W)), UNS),
        ("encode_frame16", "null planes", dict(planes=None), INV),
        ("encode_frame16", "bit_depth 8", dict(bd=8), INV),
        ("encode_frame16", "bit_depth 17", dict(bd=17), INV),
        ("encode_frame16", "odd plane pointer", dict(offsets=(1, 0, 0)), INV),
        ("encode_frame16", "odd stride", dict(strides=(2 * W + 1, W, W)), INV),
        ("encode_frame16", "short stride", dict(strides=(2 * W - 2, W, W)), INV),
        ("encode_frame16", "wider than the maximum", dict(w=2 * W, strides=(4 * W, 2 * W, 2 * W)), UNS),
    ]
    return cases


def _info_bytes(e, slot, frame):
    info = e.frame_info(slot, frame)
    return C.string_at(C.addressof(info), C.sizeof(info))


def test_malformed_submits_leave_the_slot_as_it_was():
    import h2j_b200

    env = Env()
    with h2j_b200.Encoder(max_width=W, max_height=H, max_batch=B, n_slots=2) as e:
        calls = submits(e, env)
        # the previous batch: a list of two frames of different sizes, so that frame_info differs per frame
        prev = _descs([env.p, env.p + STRIDE], W, H, W, W // 2, W * H, W * H + (W // 2) * (H // 2))
        prev[1].width, prev[1].height, prev[1].y_pitch, prev[1].c_pitch = 48, 16, 48, 24
        prev[1].u_offset, prev[1].v_offset = 48 * 16, 48 * 16 + 24 * 8

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
        for name, what, kw, status in malformed_cases():
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
