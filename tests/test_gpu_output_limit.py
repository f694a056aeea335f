"""max_jpeg_bytes is an exact limit: a JPEG of exactly max_jpeg_bytes bytes is delivered, one byte more fails with
H2J_ERR_OUTPUT_TOO_SMALL, through h2j_collect, h2j_collect_device and h2j_encode_frame alike, and no byte at or past the
limit is written.  The per-frame output stride stays a multiple of 16, so the interesting caps are the ones that the
rounding to 16 would lift to or past the JPEG's size."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W, H = 64, 48


@pytest.fixture(scope="module")
def frames(orc):
    """(planes, JPEG) of a frame whose JPEG size N has r = N mod 16 >= 2, and two neighbours that fit below N - r + 1."""
    for seed in range(100):
        p = orc.synth_planes(W, H, "textured", seed=seed, amp=40)
        jpeg = orc.oracle_encode(*p)[0]
        if len(jpeg) % 16 >= 2:
            break
    n, r = len(jpeg), len(jpeg) % 16
    assert r >= 2
    small = [orc.synth_planes(W, H, "const", seed=1, amp=0), orc.synth_planes(W, H, "textured", seed=1000, amp=10)]
    small = [(p, orc.oracle_encode(*p)[0]) for p in small]
    assert all(len(j) < n - r + 1 for _, j in small)
    return (p, jpeg), small


def _caps(n):
    r = n % 16
    return [(n, True), (n - 1, False), (n - r + 1, False)]


def test_collect_honours_the_exact_limit(orc, frames):
    import h2j_b200

    (p, want), small = frames
    batch = np.stack([orc.pack_i420(*small[0][0]), orc.pack_i420(*p), orc.pack_i420(*small[1][0])])
    for cap, fits in _caps(len(want)):
        with h2j_b200.Encoder(max_width=W, max_height=H, max_batch=3, n_slots=1, max_jpeg_bytes=cap) as e:
            e.submit_host(0, batch.ctypes.data, batch.shape[1], 3, W, H)
            res = e.collect(0, strict=False)
            assert res.status == [0, 0 if fits else h2j_b200.ERR_OUTPUT_TOO_SMALL, 0], cap
            assert res.jpegs[1] == (want if fits else b""), cap
            assert res.jpegs[0] == small[0][1] and res.jpegs[2] == small[1][1], cap


def test_collect_device_honours_the_exact_limit_and_writes_nothing_past_it(orc, frames):
    import h2j_b200

    (p, want), small = frames
    fit = np.stack([orc.pack_i420(*small[0][0]), orc.pack_i420(*small[1][0])])
    batch = np.stack([orc.pack_i420(*small[0][0]), orc.pack_i420(*p)])
    for cap, fits in _caps(len(want)):
        with h2j_b200.Encoder(max_width=W, max_height=H, max_batch=2, n_slots=1, max_jpeg_bytes=cap) as e:
            # first a batch whose JPEGs stay well below the limit: what frame 1's output holds from `cap` on, it leaves alone
            e.submit_host(0, fit.ctypes.data, fit.shape[1], 2, W, H)
            d_out, stride, sizes, st = e.collect_device(0)
            assert stride % 16 == 0 and stride >= cap and list(st) == [0, 0]
            tail = e.read_device(d_out + stride + cap, stride - cap) if stride > cap else b""
            e.submit_host(0, batch.ctypes.data, batch.shape[1], 2, W, H)
            if fits:
                d_out2, _, sizes, st = e.collect_device(0)
                assert d_out2 == d_out and list(st) == [0, 0] and int(sizes[1]) == len(want)
            else:
                with pytest.raises(h2j_b200.H2JError) as ei:
                    e.collect_device(0)
                assert ei.value.status == h2j_b200.ERR_OUTPUT_TOO_SMALL, cap
            assert e.read_device(d_out, len(small[0][1])) == small[0][1], cap
            k = min(cap, len(want) - 2)  # (EOI is written only when it fits)
            assert e.read_device(d_out + stride, k) == want[:k], cap  # the bytes below the limit are the JPEG's ...
            if stride > cap:  # ... and none at or past it was written
                assert e.read_device(d_out + stride + cap, stride - cap) == tail, cap


def test_single_frame_call_honours_the_exact_limit(orc, frames):
    import h2j_b200

    (p, want), _ = frames
    for cap, fits in _caps(len(want)):
        with h2j_b200.Encoder(max_width=W, max_height=H, max_batch=1, n_slots=1, max_jpeg_bytes=cap) as e:
            if fits:
                assert e.yuv2jpeg(*p) == want
            else:
                with pytest.raises(h2j_b200.H2JError) as ei:
                    e.yuv2jpeg(*p)
                assert ei.value.status == h2j_b200.ERR_OUTPUT_TOO_SMALL, cap
                # the raw call with a caller buffer far larger than the limit fails the same way
                import ctypes as C

                out = np.zeros(4 * len(want), np.uint8)
                n = C.c_size_t(0)
                planes = (C.c_void_p * 3)(*(x.ctypes.data for x in p))
                strides = (C.c_int * 3)(*(x.strides[0] for x in p))
                rc = e._lib.h2j_encode_frame(e._h, planes, strides, W, H, out.ctypes.data, out.size, C.byref(n))
                assert rc == h2j_b200.ERR_OUTPUT_TOO_SMALL, cap
                assert not out.any(), cap


def test_cap_smaller_than_the_header(orc, frames):
    import h2j_b200

    (p, want), small = frames
    cap = 100  # the picture header alone is ~600 bytes (DQT 69, DHT ~450)
    info_hdr = None
    batch = np.stack([orc.pack_i420(*p), orc.pack_i420(*small[0][0])])
    with h2j_b200.Encoder(max_width=W, max_height=H, max_batch=2, n_slots=1, max_jpeg_bytes=cap) as e:
        e.submit_host(0, batch.ctypes.data, batch.shape[1], 2, W, H)
        res = e.collect(0, strict=False)
        assert res.status == [h2j_b200.ERR_OUTPUT_TOO_SMALL] * 2 and res.jpegs == [b"", b""]
        info_hdr = e.frame_info(0, 0).header_bytes
        with pytest.raises(h2j_b200.H2JError) as ei:
            e.yuv2jpeg(*p)
        assert ei.value.status == h2j_b200.ERR_OUTPUT_TOO_SMALL
    assert info_hdr > cap
