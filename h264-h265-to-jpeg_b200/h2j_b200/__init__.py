"""ctypes binding of the h2j_b200 C ABI (include/h2j_b200.h).

This is the thin Python face used by tests/, bench.py and __graft_entry__.py.  It loads the in-tree
``h264-h265-to-jpeg_b200/lib/libh2j_b200.so`` (built by ``__graft_entry__.build()``) and fails loudly when the
library is missing or no CUDA device is usable -- there is no CPU path behind this module.

Reference surface being replaced: ``Encoder::yuv2Jpeg`` (reference src/Encoder.cpp:104) -- see
``Encoder.yuv2jpeg`` below for the same call shape on numpy planes.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# H2J_B200_LIB selects another build of the same library (kernel tuning experiments); there is still no fallback.
LIB_PATH = os.environ.get("H2J_B200_LIB") or os.path.join(os.path.dirname(_HERE), "lib", "libh2j_b200.so")

OK = 0
ERR_INVALID_ARG = -1
ERR_CUDA = -2
ERR_UNSUPPORTED = -3
ERR_OUTPUT_TOO_SMALL = -4
ERR_BUSY = -5
ERR_NOMEM = -6
ERR_BUFFER_TOO_SMALL = -7

RANGE_PASSTHROUGH = 0
RANGE_LIMITED_TO_FULL = 1

CHROMA_420 = 0  # what the reference opens its encoder as (src/Encoder.cpp:162)
CHROMA_422 = 1
CHROMA_444 = 2


def chroma_shape(width: int, height: int, chroma_format: int = CHROMA_420) -> Tuple[int, int]:
    """(rows, columns) of a chroma plane of a width x height frame"""
    hs = 0 if chroma_format == CHROMA_444 else 1
    vs = 1 if chroma_format == CHROMA_420 else 0
    return (height + (1 << vs) - 1) >> vs, (width + (1 << hs) - 1) >> hs


class H2JError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"h2j_b200 error {status}: {message}")
        self.status = status


class Settings(C.Structure):
    _fields_ = [
        ("device", C.c_int),
        ("max_width", C.c_int),
        ("max_height", C.c_int),
        ("max_batch", C.c_int),
        ("n_slots", C.c_int),
        ("range_mode", C.c_int),
        ("fixed_qscale", C.c_int),
        ("max_jpeg_bytes", C.c_size_t),
        ("comment", C.c_char_p),
        ("profile", C.c_int),
        ("chroma_format", C.c_int),
    ]


LAYOUT_PLANAR = 0
LAYOUT_SEMIPLANAR = 1

# h2j_rgb_format: what submit_device_rgb / rgb2jpeg take
RGB_RGB24 = 0   # R G B, 3 bytes per pixel (numpy / torch HWC)
RGB_BGR24 = 1   # B G R (OpenCV)
RGB_RGBX = 2    # R G B + one ignored byte (RGBA8)
RGB_BGRX = 3    # B G R + one ignored byte (BGRA8)
RGB_PLANAR = 4  # three planes R, G, B (torch CHW)

# h2j_resize_filter: what submit_device_resized takes (Pillow's Image.BOX, BILINEAR, BICUBIC)
FILTER_BOX = 0
FILTER_BILINEAR = 1
FILTER_BICUBIC = 2


class FrameDesc(C.Structure):
    """h2j_frame_desc: one device frame of a list submit (pitches and offsets in bytes)"""
    _fields_ = [
        ("data", C.c_void_p),
        ("width", C.c_int),
        ("height", C.c_int),
        ("y_pitch", C.c_int),
        ("c_pitch", C.c_int),
        ("u_offset", C.c_size_t),
        ("v_offset", C.c_size_t),
    ]


class FrameInfo(C.Structure):
    _fields_ = [
        ("qscale", C.c_int),
        ("mb_var_sum", C.c_int64),
        ("mcu_w", C.c_int),
        ("mcu_h", C.c_int),
        ("header_bytes", C.c_int),
        ("scan_bits", C.c_int64),
        ("stuffed_ff", C.c_int64),
        ("intra_matrix", C.c_uint8 * 64),
        ("hist", (C.c_uint32 * 256) * 4),
        ("bits", (C.c_uint8 * 17) * 4),
        ("vals", (C.c_uint8 * 256) * 4),
        ("nvals", C.c_int * 4),
    ]


EXPORTS = [
    "h2j_default_settings", "h2j_create", "h2j_destroy", "h2j_last_error", "h2j_status_string", "h2j_abi_version",
    "h2j_encode_frame", "h2j_submit_host", "h2j_submit_device", "h2j_submit_device_nv12",
    "h2j_submit_device_semiplanar", "h2j_submit_device_pitched", "h2j_collect", "h2j_collect_device", "h2j_wait",
    "h2j_alloc_pinned", "h2j_free_pinned", "h2j_convert_pad", "h2j_debug_frame_info", "h2j_debug_coefficients",
    "h2j_slot_kernel_ms", "h2j_set_profile", "h2j_slot_total_ms", "h2j_kernel_launches", "h2j_slot_set_stream",
    "h2j_slot_wait_event", "h2j_device_count", "h2j_debug_set_knob", "h2j_debug_read_device", "h2j_stream_copy",
    "h2j_submit_device_semiplanar16", "h2j_submit_device_pitched16", "h2j_encode_frame16", "h2j_submit_device_list",
    "h2j_submit_host_list", "h2j_submit_device_downscaled", "h2j_submit_device_rgb", "h2j_encode_frame_rgb",
    "h2j_debug_frame_planes", "h2j_submit_device_resized",
]

_lib = None


def load_library() -> C.CDLL:
    """dlopen the C-ABI library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
            "h2j_b200 has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    vp, ci, sz = C.c_void_p, C.c_int, C.c_size_t
    lib.h2j_default_settings.argtypes = [C.POINTER(Settings)]
    lib.h2j_default_settings.restype = None
    lib.h2j_create.argtypes = [C.POINTER(Settings), C.POINTER(vp)]
    lib.h2j_destroy.argtypes = [vp]
    lib.h2j_destroy.restype = None
    lib.h2j_last_error.argtypes = [vp]
    lib.h2j_last_error.restype = C.c_char_p
    lib.h2j_status_string.argtypes = [ci]
    lib.h2j_status_string.restype = C.c_char_p
    lib.h2j_abi_version.restype = ci
    lib.h2j_encode_frame.argtypes = [vp, C.POINTER(vp), C.POINTER(ci), ci, ci, vp, sz, C.POINTER(sz)]
    lib.h2j_submit_host.argtypes = [vp, ci, vp, sz, ci, ci, ci]
    lib.h2j_submit_device.argtypes = [vp, ci, vp, sz, ci, ci, ci]
    lib.h2j_submit_device_nv12.argtypes = [vp, ci, vp, sz, ci, sz, ci, ci, ci]
    lib.h2j_submit_device_semiplanar.argtypes = [vp, ci, vp, sz, ci, sz, ci, ci, ci]
    lib.h2j_submit_device_pitched.argtypes = [vp, ci, vp, sz, ci, ci, sz, sz, ci, ci, ci]
    lib.h2j_submit_device_semiplanar16.argtypes = [vp, ci, vp, sz, ci, sz, ci, ci, ci, ci]
    lib.h2j_submit_device_pitched16.argtypes = [vp, ci, vp, sz, ci, ci, sz, sz, ci, ci, ci, ci]
    lib.h2j_encode_frame16.argtypes = [vp, C.POINTER(vp), C.POINTER(ci), ci, ci, ci, vp, sz, C.POINTER(sz)]
    lib.h2j_submit_device_list.argtypes = [vp, ci, ci, C.POINTER(FrameDesc), ci]
    lib.h2j_submit_host_list.argtypes = [vp, ci, C.POINTER(vp), C.POINTER(ci), C.POINTER(ci), ci]
    lib.h2j_submit_device_downscaled.argtypes = [vp, ci, ci, C.POINTER(FrameDesc), ci, ci]
    lib.h2j_submit_device_resized.argtypes = [vp, ci, ci, C.POINTER(FrameDesc), ci, C.POINTER(ci), C.POINTER(ci), ci]
    lib.h2j_submit_device_rgb.argtypes = [vp, ci, ci, C.POINTER(FrameDesc), ci]
    lib.h2j_encode_frame_rgb.argtypes = [vp, ci, C.POINTER(vp), C.POINTER(ci), ci, ci, vp, sz, C.POINTER(sz)]
    lib.h2j_debug_frame_planes.argtypes = [vp, ci, ci, vp, vp, vp]
    lib.h2j_collect.argtypes = [vp, ci, vp, sz, C.POINTER(sz), C.POINTER(ci)]
    lib.h2j_collect_device.argtypes = [vp, ci, C.POINTER(vp), C.POINTER(sz), C.POINTER(sz), C.POINTER(ci)]
    lib.h2j_wait.argtypes = [vp, ci]
    lib.h2j_slot_set_stream.argtypes = [vp, ci, vp]
    lib.h2j_slot_wait_event.argtypes = [vp, ci, vp]
    lib.h2j_device_count.restype = ci
    lib.h2j_debug_set_knob.argtypes = [vp, C.c_char_p, ci]
    lib.h2j_debug_read_device.argtypes = [vp, vp, vp, sz]
    lib.h2j_alloc_pinned.argtypes = [sz]
    lib.h2j_alloc_pinned.restype = vp
    lib.h2j_free_pinned.argtypes = [vp]
    lib.h2j_free_pinned.restype = None
    lib.h2j_convert_pad.argtypes = [vp, C.POINTER(vp), C.POINTER(ci), ci, ci, ci, vp, vp, vp]
    lib.h2j_debug_frame_info.argtypes = [vp, ci, ci, C.POINTER(FrameInfo)]
    lib.h2j_debug_coefficients.argtypes = [vp, ci, ci, vp, sz]
    lib.h2j_slot_kernel_ms.argtypes = [vp, ci, C.POINTER(C.c_char_p), C.POINTER(C.c_float), ci]
    lib.h2j_set_profile.argtypes = [vp, ci]
    lib.h2j_slot_total_ms.argtypes = [vp, ci, C.POINTER(C.c_float)]
    lib.h2j_kernel_launches.argtypes = [vp]
    lib.h2j_kernel_launches.restype = C.c_longlong
    _lib = lib
    return lib


def frame_bytes(width: int, height: int, chroma_format: int = CHROMA_420) -> int:
    """Bytes of one tightly packed planar frame (Y, U, V; I420 by default)."""
    ch, cw = chroma_shape(width, height, chroma_format)
    return width * height + 2 * cw * ch


def downscaled_size(width: int, height: int, factor: int) -> Tuple[int, int]:
    """(width, height) of the frame h2j_submit_device_downscaled encodes for a width x height source at 1/factor"""
    if factor not in (2, 4, 8):
        raise ValueError(f"factor {factor} is not 2, 4 or 8")
    return (width + factor - 1) // factor, (height + factor - 1) // factor


def split_planes(frame: np.ndarray, width: int, height: int, chroma_format: int = CHROMA_420) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    ch, cw = chroma_shape(width, height, chroma_format)
    y = frame[: width * height].reshape(height, width)
    u = frame[width * height: width * height + cw * ch].reshape(ch, cw)
    v = frame[width * height + cw * ch: width * height + 2 * cw * ch].reshape(ch, cw)
    return y, u, v


def shard_range(n_items: int, rank: int, world: int) -> Tuple[int, int]:
    """Per-image sharding of a job over the ranks of one box: the half-open range of item indices rank `rank` owns.
    Images are independent, so this is the whole multi-GPU plan -- no collective touches the data path.  The first
    ``n_items % world`` ranks take one extra item; ranges are contiguous, disjoint and cover [0, n_items)."""
    if world < 1 or not (0 <= rank < world) or n_items < 0:
        raise ValueError(f"bad shard request: n_items={n_items} rank={rank} world={world}")
    base, extra = divmod(n_items, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def weighted_shards(n_items: int, weights: Sequence[float], granule: int = 1) -> List[Tuple[int, int]]:
    """Per-image sharding with shares in proportion to `weights` -- e.g. each GPU's measured host->device rate when the
    job is fed from host memory and the links of a box are not equal.  Returns one half-open range per rank: contiguous,
    disjoint, covering [0, n_items), every share a multiple of `granule` (the submit size) except that the last rank
    takes the remainder, no share empty while items are left.  Equal weights reproduce shard_range() for n_items divisible
    by len(weights) * granule."""
    k = len(weights)
    if k < 1 or n_items < 0 or granule < 1 or any(not (w > 0) for w in weights):
        raise ValueError(f"bad weighted shard request: n_items={n_items} weights={list(weights)} granule={granule}")
    total = float(sum(weights))
    units = n_items // granule  # whole granules to hand out; the remainder rides with the last rank
    shares = [int(units * w / total) for w in weights]
    # largest remainders first, so that the shares add up
    order = sorted(range(k), key=lambda i: -(units * weights[i] / total - shares[i]))
    for i in order[: units - sum(shares)]:
        shares[i] += 1
    if units >= k:  # nobody idle: take from the largest share
        for i in range(k):
            while shares[i] == 0:
                j = max(range(k), key=lambda x: shares[x])
                shares[j] -= 1
                shares[i] += 1
    out, lo = [], 0
    for i, sh in enumerate(shares):
        hi = lo + sh * granule + (n_items - units * granule if i == k - 1 else 0)
        out.append((lo, hi))
        lo = hi
    return out


def sub_batches(lo: int, hi: int, max_batch: int) -> List[Tuple[int, int]]:
    """Cut a rank's range into submit-sized pieces (each at most `max_batch` frames), in order."""
    if max_batch < 1:
        raise ValueError("max_batch must be >= 1")
    return [(s, min(s + max_batch, hi)) for s in range(lo, hi, max_batch)]


class PinnedBuffer:
    """Page-locked host memory exposed as a numpy uint8 array."""

    def __init__(self, nbytes: int):
        lib = load_library()
        self._ptr = lib.h2j_alloc_pinned(nbytes)
        if not self._ptr:
            raise H2JError(ERR_NOMEM, f"cudaHostAlloc({nbytes}) failed")
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(self._ptr))

    @property
    def ptr(self) -> int:
        return self._ptr

    def free(self) -> None:
        if self._ptr:
            self.array = None
            load_library().h2j_free_pinned(self._ptr)
            self._ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


@dataclass
class BatchResult:
    jpegs: List[bytes]
    status: List[int]


class Encoder:
    """GPU JPEG encoder.  ``yuv2jpeg`` mirrors reference ``Encoder::yuv2Jpeg`` (src/Encoder.cpp:104)."""

    def __init__(self, max_width: int = 1920, max_height: int = 1088, max_batch: int = 16, n_slots: int = 2, device: int = 0,
                 range_mode: int = RANGE_PASSTHROUGH, fixed_qscale: int = 0, max_jpeg_bytes: int = 0,
                 comment: Optional[bytes] = None, profile: bool = False, chroma_format: int = CHROMA_420):
        self._lib = load_library()
        s = Settings()
        self._lib.h2j_default_settings(C.byref(s))
        s.device, s.max_width, s.max_height, s.max_batch, s.n_slots = device, max_width, max_height, max_batch, n_slots
        s.range_mode, s.fixed_qscale, s.max_jpeg_bytes = range_mode, fixed_qscale, max_jpeg_bytes
        s.comment = comment
        s.profile = 1 if profile else 0
        s.chroma_format = chroma_format
        self.chroma_format = chroma_format
        self._h = C.c_void_p()
        rc = self._lib.h2j_create(C.byref(s), C.byref(self._h))
        if rc != OK:
            raise H2JError(rc, (self._lib.h2j_last_error(None) or b"").decode())
        self.max_batch, self.n_slots = max_batch, n_slots
        self.out_capacity = (max_jpeg_bytes or 2 * 1024 * 1024)
        self._n_in_slot = [0] * n_slots

    # -- plumbing -------------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) and self._h.value:
            self._lib.h2j_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc: int) -> None:
        if rc < 0:
            raise H2JError(rc, (self._lib.h2j_last_error(self._h) or b"").decode())

    def _check_chroma(self, w: int, h: int, u: np.ndarray, v: np.ndarray) -> None:
        want = chroma_shape(w, h, self.chroma_format)
        if u.shape != want or v.shape != want:
            raise H2JError(ERR_INVALID_ARG, f"chroma planes must be {want[0]}x{want[1]} for this encoder's chroma format, got {u.shape} / {v.shape}")

    # -- single frame, the Encoder::yuv2Jpeg shape --------------------------------------------
    def yuv2jpeg(self, y: np.ndarray, u: np.ndarray, v: np.ndarray) -> bytes:
        """One 8-bit 4:2:0 frame (2-D uint8 planes, any row stride) -> JPEG bytes."""
        for p in (y, u, v):
            if p.dtype != np.uint8 or p.ndim != 2 or p.strides[1] != 1:
                raise H2JError(ERR_INVALID_ARG, "planes must be 2-D uint8 arrays with contiguous rows")
        h, w = y.shape
        self._check_chroma(w, h, u, v)
        planes = (C.c_void_p * 3)(y.ctypes.data, u.ctypes.data, v.ctypes.data)
        strides = (C.c_int * 3)(y.strides[0], u.strides[0], v.strides[0])
        out = np.empty(self.out_capacity, np.uint8)
        n = C.c_size_t(0)
        self._check(self._lib.h2j_encode_frame(self._h, planes, strides, w, h, out.ctypes.data, out.size, C.byref(n)))
        return out[: n.value].tobytes()

    def yuv2jpeg16(self, y: np.ndarray, u: np.ndarray, v: np.ndarray, bit_depth: int) -> bytes:
        """One high-bit-depth frame (2-D uint16 planes, any row stride; `bit_depth`-bit values in the low bits of each
        little-endian word, 16 for MSB-aligned data) -> JPEG bytes of its truncated 8-bit frame (h2j_encode_frame16)."""
        for p in (y, u, v):
            if p.dtype != np.uint16 or p.ndim != 2 or p.strides[1] != 2:
                raise H2JError(ERR_INVALID_ARG, "planes must be 2-D uint16 arrays with contiguous rows")
        h, w = y.shape
        self._check_chroma(w, h, u, v)
        planes = (C.c_void_p * 3)(y.ctypes.data, u.ctypes.data, v.ctypes.data)
        strides = (C.c_int * 3)(y.strides[0], u.strides[0], v.strides[0])
        out = np.empty(self.out_capacity, np.uint8)
        n = C.c_size_t(0)
        self._check(self._lib.h2j_encode_frame16(self._h, planes, strides, bit_depth, w, h, out.ctypes.data, out.size, C.byref(n)))
        return out[: n.value].tobytes()

    def rgb2jpeg(self, image, fmt: int) -> bytes:
        """One RGB picture in host memory -> JPEG bytes (h2j_encode_frame_rgb).  Packed formats: a uint8 (H, W, 3) array
        (RGB_RGB24, RGB_BGR24) or (H, W, 4) (RGB_RGBX, RGB_BGRX) whose pixels are contiguous, at any row stride.
        RGB_PLANAR: a (3, H, W) uint8 array or three 2-D uint8 planes R, G, B, each with contiguous rows."""
        if fmt == RGB_PLANAR:
            planes = list(image)
            if len(planes) != 3 or any(p.dtype != np.uint8 or p.ndim != 2 or p.strides[1] != 1 or p.shape != planes[0].shape for p in planes):
                raise H2JError(ERR_INVALID_ARG, "planar RGB is three 2-D uint8 planes of one shape with contiguous rows")
            h, w = planes[0].shape
        else:
            bpp = 4 if fmt in (RGB_RGBX, RGB_BGRX) else 3
            if image.dtype != np.uint8 or image.ndim != 3 or image.shape[2] != bpp or image.strides[1:] != (bpp, 1):
                raise H2JError(ERR_INVALID_ARG, f"packed RGB is a uint8 (H, W, {bpp}) array with contiguous pixels")
            h, w = image.shape[:2]
            planes = [image] * 3
        ptrs = (C.c_void_p * 3)(*[p.ctypes.data for p in planes])
        strides = (C.c_int * 3)(*[p.strides[0] for p in planes])
        out = np.empty(self.out_capacity, np.uint8)
        n = C.c_size_t(0)
        self._check(self._lib.h2j_encode_frame_rgb(self._h, fmt, ptrs, strides, w, h, out.ctypes.data, out.size, C.byref(n)))
        return out[: n.value].tobytes()

    def yuv2jpeg_into(self, y: np.ndarray, u: np.ndarray, v: np.ndarray, out: Optional[np.ndarray] = None) -> int:
        """Same call, JPEG bytes into a caller buffer (or a buffer kept by this object: ``self.last_out``); returns the
        size.  Nothing is allocated per call -- the form to time."""
        if out is None:
            if getattr(self, "last_out", None) is None:
                self.last_out = np.empty(self.out_capacity, np.uint8)
            out = self.last_out
        h, w = y.shape
        planes = (C.c_void_p * 3)(y.ctypes.data, u.ctypes.data, v.ctypes.data)
        strides = (C.c_int * 3)(y.strides[0], u.strides[0], v.strides[0])
        n = C.c_size_t(0)
        self._check(self._lib.h2j_encode_frame(self._h, planes, strides, w, h, out.ctypes.data, out.size, C.byref(n)))
        return int(n.value)

    # -- batches ----------------------------------------------------------------------------------
    def submit_host(self, slot: int, frames_ptr: int, frame_stride: int, n: int, width: int, height: int) -> None:
        self._check(self._lib.h2j_submit_host(self._h, slot, frames_ptr, frame_stride, n, width, height))
        self._n_in_slot[slot] = n

    def submit_device(self, slot: int, d_frames_ptr: int, frame_stride: int, n: int, width: int, height: int) -> None:
        self._check(self._lib.h2j_submit_device(self._h, slot, d_frames_ptr, frame_stride, n, width, height))
        self._n_in_slot[slot] = n

    def submit_device_nv12(self, slot: int, d_frames_ptr: int, frame_stride: int, pitch: int, uv_offset: int, n: int,
                           width: int, height: int) -> None:
        """NV12 frames in device memory (luma plane + interleaved Cb/Cr plane, rows `pitch` apart)."""
        self._check(self._lib.h2j_submit_device_nv12(self._h, slot, d_frames_ptr, frame_stride, pitch, uv_offset, n, width, height))
        self._n_in_slot[slot] = n

    def submit_device_semiplanar(self, slot: int, d_frames_ptr: int, frame_stride: int, pitch: int, uv_offset: int, n: int,
                                 width: int, height: int) -> None:
        """Semi-planar frames in device memory by the encoder's chroma format: NV12 / NV16 / NV24 (luma plane + interleaved
        Cb/Cr plane at `uv_offset`, rows `pitch` apart)."""
        self._check(self._lib.h2j_submit_device_semiplanar(self._h, slot, d_frames_ptr, frame_stride, pitch, uv_offset, n, width, height))
        self._n_in_slot[slot] = n

    def submit_device_pitched(self, slot: int, d_frames_ptr: int, frame_stride: int, y_pitch: int, c_pitch: int, u_offset: int,
                              v_offset: int, n: int, width: int, height: int) -> None:
        """Planar frames in device memory at any layout: luma rows `y_pitch` apart at the frame's start, Cb / Cr planes at
        `u_offset` / `v_offset` with rows `c_pitch` apart."""
        self._check(self._lib.h2j_submit_device_pitched(self._h, slot, d_frames_ptr, frame_stride, y_pitch, c_pitch, u_offset, v_offset,
                                                        n, width, height))
        self._n_in_slot[slot] = n

    def submit_device_semiplanar16(self, slot: int, d_frames_ptr: int, frame_stride: int, pitch: int, uv_offset: int, bit_depth: int,
                                   n: int, width: int, height: int) -> None:
        """Semi-planar frames of 16-bit words in device memory (P010 / P016, P210 / P216, ... by the encoder's chroma
        format); pitch and offsets in bytes, `bit_depth`-bit values in the low bits of each word (16 for MSB-aligned)."""
        self._check(self._lib.h2j_submit_device_semiplanar16(self._h, slot, d_frames_ptr, frame_stride, pitch, uv_offset, bit_depth, n,
                                                             width, height))
        self._n_in_slot[slot] = n

    def submit_device_pitched16(self, slot: int, d_frames_ptr: int, frame_stride: int, y_pitch: int, c_pitch: int, u_offset: int,
                                v_offset: int, bit_depth: int, n: int, width: int, height: int) -> None:
        """Planar frames of 16-bit words in device memory at any layout (pitches and offsets in bytes)."""
        self._check(self._lib.h2j_submit_device_pitched16(self._h, slot, d_frames_ptr, frame_stride, y_pitch, c_pitch, u_offset, v_offset,
                                                          bit_depth, n, width, height))
        self._n_in_slot[slot] = n

    def submit_device_list(self, slot: int, layout: int, descs: Sequence[FrameDesc]) -> None:
        """Device frames each at its own address and of its own size (LAYOUT_PLANAR or LAYOUT_SEMIPLANAR for all)."""
        arr = (FrameDesc * max(1, len(descs)))(*descs)
        self._check(self._lib.h2j_submit_device_list(self._h, slot, layout, arr, len(descs)))
        self._n_in_slot[slot] = len(descs)

    def submit_device_downscaled(self, slot: int, layout: int, descs: Sequence[FrameDesc], factor: int) -> None:
        """Device frames as for submit_device_list, each encoded box-filtered to 1/factor (2, 4 or 8) of its size
        (downscaled_size); only the downscaled frames must fit the encoder's maximum."""
        arr = (FrameDesc * max(1, len(descs)))(*descs)
        self._check(self._lib.h2j_submit_device_downscaled(self._h, slot, layout, arr, len(descs), factor))
        self._n_in_slot[slot] = len(descs)

    def submit_device_resized(self, slot: int, layout: int, descs: Sequence[FrameDesc], sizes: Sequence[Tuple[int, int]], filter: int) -> None:
        """Device frames as for submit_device_list, frame i encoded resized to sizes[i] = (width, height) with a FILTER_* of
        Pillow's (PIL.Image.resize on every plane); only the resized frames must fit the encoder's maximum."""
        n = len(descs)
        arr = (FrameDesc * max(1, n))(*descs)
        ws = (C.c_int * max(1, len(sizes)))(*[w for w, _ in sizes])
        hs = (C.c_int * max(1, len(sizes)))(*[h for _, h in sizes])
        if len(sizes) != n:
            raise H2JError(ERR_INVALID_ARG, f"{n} frames but {len(sizes)} sizes")
        self._check(self._lib.h2j_submit_device_resized(self._h, slot, layout, arr, n, ws, hs, filter))
        self._n_in_slot[slot] = n

    def submit_device_rgb(self, slot: int, fmt: int, descs: Sequence[FrameDesc]) -> None:
        """RGB device frames (an RGB_* format for all), each at its own address and of its own size: packed formats use
        data, width, height and y_pitch; RGB_PLANAR has G at data + u_offset and B at data + v_offset, rows y_pitch apart.
        A (3, H, W) CUDA tensor t is FrameDesc(t.data_ptr(), W, H, t.stride(1), 0, t.stride(0), 2 * t.stride(0))."""
        arr = (FrameDesc * max(1, len(descs)))(*descs)
        self._check(self._lib.h2j_submit_device_rgb(self._h, slot, fmt, arr, len(descs)))
        self._n_in_slot[slot] = len(descs)

    def submit_host_list(self, slot: int, frames: Sequence[int], sizes: Sequence[Tuple[int, int]]) -> None:
        """Tight planar frames in host memory (addresses, as from ndarray.ctypes.data), each of its own (width, height)."""
        n = len(frames)
        ptrs = (C.c_void_p * max(1, n))(*frames)
        ws = (C.c_int * max(1, n))(*[w for w, _ in sizes])
        hs = (C.c_int * max(1, n))(*[h for _, h in sizes])
        self._check(self._lib.h2j_submit_host_list(self._h, slot, ptrs, ws, hs, n))
        self._n_in_slot[slot] = n

    def read_device(self, d_ptr: int, nbytes: int) -> bytes:
        """Bytes of device memory on the encoder's device (e.g. one JPEG left there by collect_device)."""
        out = np.empty(nbytes, np.uint8)
        self._check(self._lib.h2j_debug_read_device(self._h, d_ptr, out.ctypes.data, nbytes))
        return out.tobytes()

    def set_knob(self, name: str, value: int) -> None:
        """Launch-shape override for tests (h2j_debug_set_knob); results never depend on it."""
        self._check(self._lib.h2j_debug_set_knob(self._h, name.encode(), value))

    def set_profile(self, on: bool) -> None:
        """Per-kernel event brackets for the batches submitted from now on."""
        self._check(self._lib.h2j_set_profile(self._h, 1 if on else 0))

    def set_stream(self, slot: int, cuda_stream: int) -> None:
        """Enqueue the slot's work on a caller-owned stream (raw cudaStream_t handle)."""
        self._check(self._lib.h2j_slot_set_stream(self._h, slot, cuda_stream))

    def wait_event(self, slot: int, cuda_event: int) -> None:
        """Order the slot's next work behind a CUDA event (raw cudaEvent_t, e.g. ``torch.cuda.Event().cuda_event``)
        recorded behind whatever produces the next batch's device input."""
        self._check(self._lib.h2j_slot_wait_event(self._h, slot, cuda_event))

    def wait(self, slot: int) -> None:
        self._check(self._lib.h2j_wait(self._h, slot))

    def collect_into(self, slot: int, out_ptr: int, out_capacity: int, strict: bool = True) -> Tuple[np.ndarray, np.ndarray]:
        """Copy the slot's JPEGs packed into caller memory; returns (offsets[n+1], status[n]).  A frame that failed has
        length 0 and a non-zero status; with strict=True (default) that raises, the good frames are still in the buffer.
        ERR_BUFFER_TOO_SMALL (caller buffer short) leaves the slot collectable: H2JError.offsets holds the sizes."""
        n = self._n_in_slot[slot]
        offs = (C.c_size_t * (n + 1))()
        st = (C.c_int * n)()
        rc = self._lib.h2j_collect(self._h, slot, out_ptr, out_capacity, offs, st)
        offsets, status = np.frombuffer(offs, dtype=np.uintp).copy(), np.frombuffer(st, dtype=np.intc).copy()
        if rc == ERR_BUFFER_TOO_SMALL or (rc < 0 and (strict or not status.any())):
            err = H2JError(rc, (self._lib.h2j_last_error(self._h) or b"").decode())
            err.offsets, err.frame_status = offsets, status
            raise err
        return offsets, status

    def collect(self, slot: int, strict: bool = True) -> BatchResult:
        n = self._n_in_slot[slot]
        out = np.empty((self.out_capacity + 15) // 16 * 16 * n, np.uint8)
        offs, st = self.collect_into(slot, out.ctypes.data, out.size, strict=strict)
        return BatchResult([out[int(offs[i]): int(offs[i + 1])].tobytes() for i in range(n)], [int(x) for x in st])

    def collect_device(self, slot: int) -> Tuple[int, int, np.ndarray, np.ndarray]:
        """Leave the JPEGs on the device: returns (device pointer, per-frame capacity, sizes, status)."""
        n = self._n_in_slot[slot]
        d_out = C.c_void_p()
        cap = C.c_size_t()
        sizes = (C.c_size_t * n)()
        st = (C.c_int * n)()
        self._check(self._lib.h2j_collect_device(self._h, slot, C.byref(d_out), C.byref(cap), sizes, st))
        return d_out.value, cap.value, np.frombuffer(sizes, dtype=np.uintp).copy(), np.frombuffer(st, dtype=np.intc).copy()

    def encode_batch(self, frames: np.ndarray, width: int, height: int, slot: int = 0) -> BatchResult:
        """frames: (n, frame_bytes) uint8 host array of tight I420 frames."""
        assert frames.dtype == np.uint8 and frames.ndim == 2 and frames.flags.c_contiguous
        self.submit_host(slot, frames.ctypes.data, frames.shape[1], frames.shape[0], width, height)
        return self.collect(slot)

    # -- kernel 1 on its own -----------------------------------------------------------------
    def convert_pad(self, y: np.ndarray, u: np.ndarray, v: np.ndarray, range_mode: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        h, w = y.shape
        self._check_chroma(w, h, u, v)
        mw, mh = (w + 15) // 16, (h + 15) // 16
        oy = np.empty((mh * 16, mw * 16), np.uint8)
        ou = np.empty((mh * 8, mw * 8), np.uint8)
        ov = np.empty((mh * 8, mw * 8), np.uint8)
        planes = (C.c_void_p * 3)(y.ctypes.data, u.ctypes.data, v.ctypes.data)
        strides = (C.c_int * 3)(y.strides[0], u.strides[0], v.strides[0])
        self._check(self._lib.h2j_convert_pad(self._h, planes, strides, w, h, range_mode, oy.ctypes.data, ou.ctypes.data, ov.ctypes.data))
        return oy, ou, ov

    # -- inspection ---------------------------------------------------------------------------
    def frame_info(self, slot: int, frame: int) -> FrameInfo:
        info = FrameInfo()
        self._check(self._lib.h2j_debug_frame_info(self._h, slot, frame, C.byref(info)))
        return info

    def coefficients(self, slot: int, frame: int, n_blocks: int) -> np.ndarray:
        out = np.empty((n_blocks, 64), np.int16)
        self._check(self._lib.h2j_debug_coefficients(self._h, slot, frame, out.ctypes.data, out.size))
        return out

    def frame_planes(self, slot: int, frame: int, width: int, height: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """(y, u, v) of frame `frame` of the slot's last batch as the pipeline read it (h2j_debug_frame_planes); width x
        height is that frame's size as encoded (a downscaled frame's: downscaled_size)."""
        # the hook writes the frame's own size: buffers large enough for any frame of the MCU geometry the slot reports
        info = self.frame_info(slot, frame)
        mcu_px = 8 if self.chroma_format == CHROMA_444 else 16
        if (info.mcu_w, info.mcu_h) != (-(-width // mcu_px), -(-height // 16)):
            raise H2JError(ERR_INVALID_ARG, f"frame {frame} of slot {slot} is not {width}x{height}")
        bw, bh = info.mcu_w * mcu_px, info.mcu_h * 16
        bch, bcw = chroma_shape(bw, bh, self.chroma_format)
        y, u, v = np.empty(bw * bh, np.uint8), np.empty(bch * bcw, np.uint8), np.empty(bch * bcw, np.uint8)
        self._check(self._lib.h2j_debug_frame_planes(self._h, slot, frame, y.ctypes.data, u.ctypes.data, v.ctypes.data))
        ch, cw = chroma_shape(width, height, self.chroma_format)
        return y[: width * height].reshape(height, width), u[: cw * ch].reshape(ch, cw), v[: cw * ch].reshape(ch, cw)

    def kernel_ms(self, slot: int) -> List[Tuple[str, float]]:
        names = (C.c_char_p * 32)()
        ms = (C.c_float * 32)()
        n = self._lib.h2j_slot_kernel_ms(self._h, slot, names, ms, 32)
        self._check(n)
        return [(names[i].decode(), float(ms[i])) for i in range(n)]

    def total_ms(self, slot: int) -> float:
        ms = C.c_float()
        self._check(self._lib.h2j_slot_total_ms(self._h, slot, C.byref(ms)))
        return float(ms.value)

    @property
    def kernel_launches(self) -> int:
        return int(self._lib.h2j_kernel_launches(self._h))
