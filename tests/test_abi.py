"""CPU suite: the C-ABI library loads, exports every symbol include/h2j_b200.h declares, and fails LOUDLY
without a CUDA device (no CPU fallback).  No compute calls here."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    h = open(os.path.join(ROOT, "include", "h2j_b200.h")).read()
    h = re.sub(r"/\*.*?\*/", "", h, flags=re.S)
    return sorted(set(re.findall(r"\b(h2j_[a-z0-9_]+)\s*\(", h)))


def test_every_declared_symbol_is_exported():
    import h2j_b200

    lib = h2j_b200.load_library()
    names = _declared()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/h2j_b200.h but not exported"
    assert set(h2j_b200.EXPORTS) <= set(names)
    assert lib.h2j_abi_version() == 3


def test_status_strings_and_defaults():
    import h2j_b200

    lib = h2j_b200.load_library()
    s = h2j_b200.Settings()
    lib.h2j_default_settings(C.byref(s))
    assert (s.max_width, s.max_height, s.range_mode, s.fixed_qscale, s.chroma_format) == (1920, 1088, 0, 0, 0)
    import ctypes

    # the binding's struct is the header's struct (a field appended in C without the Python side following would shift nothing
    # visible here but truncate the copy in h2j_create)
    hdr = open(os.path.join(ROOT, "include", "h2j_b200.h")).read()
    body = hdr[hdr.index("typedef struct h2j_settings {"): hdr.index("} h2j_settings;")]
    fields = re.findall(r"^\s+(?:const\s+)?(?:int|size_t|char)\s*\*?\s*(\w+);", body, flags=re.M)
    assert fields == [f[0] for f in h2j_b200.Settings._fields_], fields
    assert lib.h2j_status_string(0) == b"ok"
    assert b"CUDA" in lib.h2j_status_string(-2)


def test_bad_settings_rejected():
    import h2j_b200

    with pytest.raises(h2j_b200.H2JError) as ei:
        h2j_b200.Encoder(max_width=1, max_height=1)
    assert ei.value.status == h2j_b200.ERR_INVALID_ARG
    # a comment whose COM segment length (text + NUL + 2) does not fit 16 bits; checked before any device is looked for
    with pytest.raises(h2j_b200.H2JError) as ei:
        h2j_b200.Encoder(comment=b"c" * 65533)
    assert ei.value.status == h2j_b200.ERR_INVALID_ARG and "COM segment" in str(ei.value)


def test_no_gpu_means_loud_failure():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import h2j_b200

    with pytest.raises(h2j_b200.H2JError) as ei:
        h2j_b200.Encoder()
    assert ei.value.status == h2j_b200.ERR_CUDA
    assert "no CPU path" in str(ei.value)


def test_product_sources_do_not_touch_the_oracle():
    """The product path (package + include) must not reference oracle/ or the reference tree."""
    pkg = os.path.join(ROOT, "h264-h265-to-jpeg_b200")
    for base, _, files in os.walk(pkg):
        if os.sep + "lib" in base:
            continue
        for f in files:
            if f.endswith((".cu", ".cuh", ".cpp", ".h", ".py")):
                txt = open(os.path.join(base, f), errors="ignore").read()
                assert "mjpeg_oracle" not in txt and "libh2j_oracle" not in txt and "libh2j_ref" not in txt, f
