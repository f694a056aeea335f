"""GPU suite: the launch shapes the throughput runs use, on geometries that do not divide into whole tiles.

K2 (fdct_quant_kernel) lets one CTA walk several consecutive 16-MCU tiles when the batch is large (16 at the bench's
2048 frames): chroma DC carried from tile to tile, block positions advanced across MCU-row ends, bulk stores of one tile
under the transform of the next.  Small test batches would never take that loop, so it is forced here
(h2j_debug_set_knob) on frames whose last tile and last 32-block unit are partial, with batches of 8, planar and NV12
read in place, every JPEG compared with the oracle byte for byte.  Then the bench's other geometries (configs[3]: 4K and
1918x1078) at real batch sizes with a sample of frames compared."""
import numpy as np
import pytest

from tests.support.layouts import place, upload

pytestmark = pytest.mark.gpu


# (w, h): MCUs -> tiles.  641x479: 41x30 = 1230 -> 76.9 (last tile 14 MCUs, last unit 20 blocks); 330x225: 21x15 = 315 ->
# 19.7; 330x241: 21x16 = 336 -> 21 (whole tiles, odd sizes); 17x4098: 2x257 = 514 -> 32.1 (two MCUs per row: every tile spans
# eight MCU rows, the last one holds 2 MCUs); 2562x1442: 161x91 = 14651 -> 915.7
@pytest.mark.parametrize("w,h", [(641, 479), (330, 225), (330, 241), (17, 4098), (2562, 1442)])
def test_multi_tile_ctas_on_partial_tiles(orc, w, h):
    import h2j_b200

    n = 8
    planes = [orc.synth_planes(w, h, "textured" if s % 3 else "noise", seed=300 + s, amp=12 + 11 * s) for s in range(n)]
    want = [orc.oracle_encode(*p)[0] for p in planes]
    frames = np.stack([orc.pack_i420(*p) for p in planes])
    stride = (frames.shape[1] + 255) // 256 * 256
    d, ptr = upload(frames, stride)
    cw = (w + 1) // 2
    pitch = (max(w, 2 * cw) + 63) // 64 * 64
    nv = [place(*p, pitch, pitch, pitch * h, size=pitch * (h + p[1].shape[0]), pad=0x5A) for p in planes]
    nstride = (len(nv[0]) + 255) // 256 * 256
    dn, nptr = upload(nv, nstride)
    with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=n, n_slots=1) as e:
        for tpc in (2, 5, 16):
            e.set_knob("fdct_tiles_per_cta", tpc)
            e.submit_device(0, ptr, stride, n, w, h)
            res = e.collect(0)
            assert res.status == [0] * n
            for i in range(n):
                assert res.jpegs[i] == want[i], f"{w}x{h}, {tpc} tiles per CTA, planar frame {i}"
            e.submit_device_nv12(0, nptr, nstride, pitch, pitch * h, n, w, h)
            res = e.collect(0)
            for i in range(n):
                assert res.jpegs[i] == want[i], f"{w}x{h}, {tpc} tiles per CTA, NV12 frame {i}"
        e.set_knob("fdct_tiles_per_cta", 0)
        # host frames through the same loop (odd widths are re-pitched on the device first)
        e.set_knob("fdct_tiles_per_cta", 3)
        assert e.encode_batch(frames, w, h).jpegs == want


@pytest.mark.parametrize("w,h,n", [(3840, 2160, 64), (1918, 1078, 256), (1920, 1080, 512)])
def test_large_batches_of_the_bench_geometries_sampled(orc, w, h, n):
    """BASELINE.json configs[3] / configs[2] shapes at the batch sizes where K2 walks several tiles per CTA by itself
    and K4b takes its 32-units-per-warp form; first, last and random frames against the oracle, all sizes sane."""
    import torch

    import bench
    import h2j_b200

    dev = torch.device("cuda", 0)
    d_frames, fb, stride = bench.make_frames_torch(n, w, h, dev, seed0=7)
    torch.cuda.synchronize()
    rng = np.random.default_rng(w + n)
    pick = sorted({0, n - 1, *[int(x) for x in rng.integers(1, n - 1, 4)]})
    with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=n, n_slots=1, max_jpeg_bytes=4 * 1024 * 1024) as e:
        e.submit_device(0, d_frames.data_ptr(), stride, n, w, h)
        d_out, cap, sizes, st = e.collect_device(0)
        assert (st == 0).all() and (sizes > 1000).all()
        for i in pick:
            got = e.read_device(d_out + i * cap, int(sizes[i]))
            y, u, v = h2j_b200.split_planes(d_frames[i, :fb].cpu().numpy(), w, h)
            want = orc.oracle_encode(np.ascontiguousarray(y), np.ascontiguousarray(u), np.ascontiguousarray(v))[0]
            assert got == want, f"{w}x{h} batch {n}: frame {i} differs from the oracle"
