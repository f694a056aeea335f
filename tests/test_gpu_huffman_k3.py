"""K3 (huffman_kernel) on its own, on 2,000 adversarial histograms (tests/support/histograms.py) sent as one batch of 500
frames, against the oracle's table builder (orc_huffman_table): BITS, HUFFVAL, the code tables K4a reads and the picture
header.  K3's tables are also checked against the tie-order-free properties of tests/test_huffman_tables.py, so that a
failure says which side is wrong."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests.support import histograms as H
from tests.test_huffman_tables import oracle_table

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
HDR_CAP = 2048
COMMENT = b"k3 shim"  # what k3_shim.cu puts into the COM segment
DQT = bytes(range(1, 65))  # ... and into the DQT payload


def _nvcc():
    for p in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if p and os.path.exists(p):
            return p
    return None


@pytest.fixture(scope="module")
def k3(tmp_path_factory):
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("the CUDA toolkit (nvcc) is not installed: the K3 shim cannot be built")
    so = str(tmp_path_factory.mktemp("k3shim") / "libk3shim.so")
    subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-shared",
                    "-o", so, os.path.join(HERE, "support", "k3_shim.cu")], check=True)
    lib = C.CDLL(so)
    vp = C.c_void_p
    lib.k3_run.argtypes = [C.c_int, vp, vp, vp, vp, vp, vp, C.c_int, vp, vp]
    return lib


@pytest.fixture(scope="module")
def run(k3):
    """The 2,000 histograms as 500 frames: two DC and two AC histograms per frame.  Returns (hist, K3 outputs)."""
    dc, ac = H.generate()
    n = len(ac) // 2
    hist = np.zeros((n, 4, 256), np.uint32)
    kinds = np.empty((n, 4), object)
    for f in range(n):
        for t, (kind, h) in zip(range(4), (dc[2 * f], dc[2 * f + 1], ac[2 * f], ac[2 * f + 1])):
            hist[f, t], kinds[f, t] = h, kind
    out = dict(bits=np.zeros((n, 4, 17), np.uint8), vals=np.zeros((n, 4, 256), np.uint8), nvals=np.zeros((n, 4), np.intc),
               hcode=np.zeros((n, 4, 256), np.uint32), hdr=np.zeros((n, HDR_CAP), np.uint8), hdr_bytes=np.zeros(n, np.intc),
               status=np.zeros(n, np.intc))
    rc = k3.k3_run(n, hist.ctypes.data, *(out[k].ctypes.data for k in ("bits", "vals", "nvals", "hcode", "hdr")), HDR_CAP,
                   out["hdr_bytes"].ctypes.data, out["status"].ctypes.data)
    assert rc == 0, f"CUDA error {rc}"
    return hist, kinds, out


def _code_table(out, f, t):
    """K3's code table of table t: 16 DC entries at hcode[1][224 + 16 * t], 256 AC entries at hcode[t]"""
    return out["hcode"][f, 1, 224 + 16 * t: 240 + 16 * t] if t < 2 else out["hcode"][f, t]


def _header(bits4, vals4, nvals4):
    """SOI, COM, DQT, DHT, SOF0 (64x48, 4:2:0), SOS as mjpegenc_common.c writes them, from the oracle's tables"""
    com = b"\xff\xfe" + (len(COMMENT) + 3).to_bytes(2, "big") + COMMENT + b"\x00"
    dqt = b"\xff\xdb\x00\x43\x00" + DQT
    sof = bytes([0xFF, 0xC0, 0, 17, 8, 0, 48, 0, 64, 3, 1, 0x22, 0, 2, 0x11, 0, 3, 0x11, 0])
    sos = bytes([0xFF, 0xDA, 0, 12, 3, 1, 0x00, 2, 0x11, 3, 0x11, 0, 63, 0])
    return b"\xff\xd8" + com + dqt + H.dht_segment(bits4, vals4, nvals4) + sof + sos


def test_k3_tables_equal_the_oracle(run, orc):
    hist, kinds, out = run
    n = hist.shape[0]
    assert (out["status"] == 0).all()
    for f in range(n):
        want = [oracle_table(orc, hist[f, t]) for t in range(4)]
        for t in range(4):
            what = (f, t, kinds[f, t])
            bits, vals, nv = want[t]
            got_bits, got_vals, got_nv = out["bits"][f, t], out["vals"][f, t], int(out["nvals"][f, t])
            # K3 on its own first: a failure here is K3's, whatever the oracle says
            bad = H.check_table(hist[f, t], got_bits, got_vals, got_nv)
            assert not bad, (what, "K3 table", bad)
            assert got_nv == nv, what
            assert bytes(got_bits) == bytes(bits), what
            assert bytes(got_vals[:nv]) == bytes(vals[:nv]), what
            # the code table K4a reads: every used symbol, and zero where nothing is used
            table = _code_table(out, f, t)
            want_tab = np.zeros(len(table), np.uint32)
            for sym, (code, length) in H.canonical_codes(bits, vals).items():
                want_tab[sym] = H.code_table_entry(sym, code, length)
            bad_syms = np.nonzero(table != want_tab)[0]
            assert bad_syms.size == 0, (what, [(int(s), hex(int(table[s])), hex(int(want_tab[s]))) for s in bad_syms[:4]])
        hdr = _header([w[0] for w in want], [w[1] for w in want], [w[2] for w in want])
        assert int(out["hdr_bytes"][f]) == len(hdr), f
        assert out["hdr"][f, : len(hdr)].tobytes() == hdr, f
        assert not out["hdr"][f, len(hdr):].any(), f
    # the parts of hcode that are not code tables stay untouched
    assert not out["hcode"][:, 0].any() and not out["hcode"][:, 1, :224].any()


def test_k3_batch_reaches_the_limits(run):
    """The batch holds what the tests above are meant to see: 1 and 256 used symbols, 16-bit codes in many tables,
    code-table entries that use all 32 bits (a 16-bit code behind 9 mantissa bits and more)."""
    hist, kinds, out = run
    used = (hist != 0).sum(axis=2)
    assert used.min() == 1 and used.max() == 256
    assert (out["bits"][:, :, 16] > 0).sum() >= 100
    full = 0
    for f in range(hist.shape[0]):
        for t in (2, 3):
            for sym, (code, length) in H.canonical_codes(out["bits"][f, t], out["vals"][f, t]).items():
                full += length == 16 and (sym & 15) == 9
    assert full >= 20
