"""ctypes binding of libvstab.so (include/vstab.h) -- the Python face of the C ABI.

`Stabilizer` mirrors class Stabilizer of the reference
(/root/reference/include/stabilizer.hpp:106-475): same constructor arguments and
defaults, `stabilize_frame`, `set_stabilization_mode`, `total_frame_window_size`,
static `decompose_homography` / `compose_homography`, and the reference's error
behaviour (std::invalid_argument -> ValueError).  There is no CPU fallback: if
the shared library is missing or no sm_100 device is present the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

ACCUMULATED_FULL_LOCK, ORB_FULL_LOCK, SIFT_FULL_LOCK, TRANSLATION_LOCK, ROTATION_LOCK, GLOBAL_SMOOTHING = range(6)

OK, ERR_INVALID_ARGUMENT, ERR_SIZE_CHANGED, ERR_CUDA, ERR_UNSUPPORTED, ERR_STATE, ERR_NCCL = range(7)
SRC_HOST, SRC_SIMULATOR, SRC_DEVICE = 0, 1, 2
PIX_NV12, PIX_I420 = 1, 2

TAP_GRAY, TAP_PYR1, TAP_PYR2, TAP_PYR3, TAP_PREV_PTS, TAP_LK_PTS, TAP_LK_STATUS, TAP_NEW_PTS, TAP_T, TAP_M, \
    TAP_H_STABILIZE, TAP_H_SCALED, TAP_BORDER, TAP_EIG, TAP_INLIERS, TAP_CHANNEL_SUMS, TAP_LOCK_H, TAP_ORB_COUNTS, \
    TAP_FEAT_GRAY = range(19)

_PKG_ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), "..", ".."))
LIB_PATH = os.path.join(_PKG_ROOT, "lib", "libvstab.so")


class VstabError(RuntimeError):
    pass


class HParams(C.Structure):
    """struct HomographyParameters, include/stabilizer.hpp:44-57"""
    _fields_ = [("s", C.c_double), ("theta", C.c_double), ("k", C.c_double), ("delta", C.c_double),
                ("t", C.c_double * 2), ("v", C.c_double * 2)]


class YuvLayout(C.Structure):          # vstab_yuv_layout: plane k at base + offset[k], rows step[k] bytes apart
    _fields_ = [("format", C.c_int), ("offset", C.c_size_t * 3), ("step", C.c_size_t * 3)]

    @classmethod
    def make(cls, fmt: int, offsets, steps):
        off, st = list(offsets) + [0] * (3 - len(offsets)), list(steps) + [0] * (3 - len(steps))
        return cls(int(fmt), (C.c_size_t * 3)(*off), (C.c_size_t * 3)(*st))


class NcclId(C.Structure):
    _fields_ = [("bytes", C.c_char * 128)]


class ShardPlan(C.Structure):
    _fields_ = [("first", C.c_long), ("last", C.c_long), ("call_first", C.c_long), ("call_last", C.c_long)]


class FusedPlan(C.Structure):           # vstab_fused_plan
    _fields_ = [("ring_chunks", C.c_long), ("fused_first", C.c_long), ("fused_last", C.c_long)]


class OfflineCfg(C.Structure):          # vstab_offline_cfg
    _fields_ = [("n_total", C.c_long), ("mode", C.c_int), ("lock_call", C.c_long), ("source", C.c_int),
                ("host_frames", C.c_void_p), ("frame_stride", C.c_size_t), ("step", C.c_size_t), ("host_halo", C.c_void_p),
                ("d_texture", C.c_void_p), ("tex_rows", C.c_int), ("tex_cols", C.c_int), ("poses", C.POINTER(C.c_double)),
                ("focal", C.c_double),
                ("host_out", C.c_void_p), ("out_frame_stride", C.c_size_t), ("out_step", C.c_size_t), ("d_out", C.c_void_p),
                ("checksums", C.POINTER(C.c_uint64)), ("T_all", C.POINTER(C.c_double))]


class OfflineReport(C.Structure):       # vstab_offline_report
    _fields_ = [("source_ms", C.c_float), ("estimate_ms", C.c_float), ("exchange_ms", C.c_float), ("render_ms", C.c_float),
                ("total_ms", C.c_float), ("frames", C.c_long), ("calls", C.c_long)]


_u8p = C.POINTER(C.c_uint8)
_f32p = C.POINTER(C.c_float)
_f64p = C.POINTER(C.c_double)
_vp = C.c_void_p

# every symbol include/vstab.h declares: (restype, argtypes)
SYMBOLS = {
    "vstab_abi_version": (C.c_int, []),
    "vstab_status_string": (C.c_char_p, [C.c_int]),
    "vstab_create": (C.c_int, [C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.POINTER(_vp)]),
    "vstab_destroy": (None, [_vp]),
    "vstab_set_mode": (C.c_int, [_vp, C.c_int]),
    "vstab_get_mode": (C.c_int, [_vp]),
    "vstab_total_frame_window_size": (C.c_size_t, [_vp]),
    "vstab_stabilize_frame": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_size_t, _vp, C.c_size_t]),
    "vstab_stabilize_frame_device": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_size_t, _vp, C.c_size_t]),
    "vstab_synchronize": (C.c_int, [_vp]),
    "vstab_yuv_layout_packed": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.POINTER(YuvLayout)]),
    "vstab_stabilize_frame_yuv": (C.c_int, [_vp, _vp, C.POINTER(YuvLayout), C.c_int, C.c_int, _vp, C.POINTER(YuvLayout)]),
    "vstab_stabilize_frame_yuv_device": (C.c_int, [_vp, _vp, C.POINTER(YuvLayout), C.c_int, C.c_int, _vp, C.POINTER(YuvLayout)]),
    "vstab_offline_set_yuv": (C.c_int, [_vp, C.POINTER(YuvLayout), C.POINTER(YuvLayout)]),
    "vstab_k_yuv_to_bgr": (C.c_int, [C.c_int, _vp, C.POINTER(YuvLayout), C.c_int, C.c_int, _vp, C.c_size_t]),
    "vstab_k_bgr_to_yuv": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int, C.c_size_t, _vp, C.POINTER(YuvLayout)]),
    "vstab_decompose_homography": (C.c_int, [_f64p, C.c_double, C.c_double, C.POINTER(HParams)]),
    "vstab_compose_homography": (None, [C.POINTER(HParams), C.c_double, C.c_double, _f64p]),
    "vstab_last_error": (C.c_char_p, [_vp]),
    "vstab_set_trail": (C.c_int, [_vp, C.c_int]),
    "vstab_set_partial_lock_fix": (C.c_int, [_vp, C.c_int]),
    "vstab_set_crop": (C.c_int, [_vp, C.c_double, C.c_double]),
    "vstab_crop_zoom": (C.c_double, [_f64p, C.c_int, C.c_int, C.c_double]),
    "vstab_offline_set_crop": (C.c_int, [_vp, C.c_double, C.c_double]),
    "vstab_k_copy_feathered": (C.c_int, [C.c_int, _vp, _vp, C.c_int, C.c_int, C.c_size_t, _f64p, _vp, C.c_size_t]),
    "vstab_host_alloc": (_vp, [C.c_size_t]),
    "vstab_host_free": (None, [_vp]),
    "vstab_read_tap": (C.c_long, [_vp, C.c_int, _vp, C.c_size_t]),
    "vstab_working_width": (C.c_int, [_vp]),
    "vstab_working_height": (C.c_int, [_vp]),
    "vstab_presentation_index": (C.c_long, [_vp]),
    "vstab_offline_create": (C.c_int, [C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    "vstab_offline_destroy": (None, [_vp]),
    "vstab_offline_estimate": (C.c_int, [_vp, _vp, C.c_size_t, C.c_size_t, C.c_int, C.c_long, _vp, _vp, _vp]),
    "vstab_offline_render": (C.c_int, [_vp, _vp, C.c_size_t, C.c_size_t, C.c_long, C.c_int, C.c_long, _vp, C.c_long,
                                       C.c_int, C.c_long, _vp, _vp, C.c_size_t, C.c_size_t]),
    "vstab_offline_run_host": (C.c_int, [_vp, _vp, C.c_size_t, C.c_size_t, C.c_long, C.c_int, C.c_long, _vp, C.c_size_t,
                                       C.c_size_t]),
    "vstab_offline_reference_bytes": (C.c_size_t, []),
    "vstab_offline_reference_capture": (C.c_int, [_vp, _vp, C.c_size_t, C.c_int]),
    "vstab_offline_reference_export": (C.c_int, [_vp, _vp]),
    "vstab_offline_reference_import": (C.c_int, [_vp, _vp, C.c_int]),
    "vstab_offline_register": (C.c_int, [_vp, _vp, C.c_size_t, C.c_size_t, C.c_int, _vp]),
    "vstab_offline_set_registrations": (C.c_int, [_vp, _vp, C.c_long]),
    "vstab_offline_synchronize": (C.c_int, [_vp]),
    "vstab_offline_last_error": (C.c_char_p, [_vp]),
    "vstab_nccl_get_unique_id": (C.c_int, [C.POINTER(NcclId)]),
    "vstab_offline_comm_init": (C.c_int, [_vp, C.POINTER(NcclId), C.c_int, C.c_int]),
    "vstab_offline_plan": (C.c_int, [C.c_long, C.c_int, C.c_int, C.c_size_t, C.POINTER(ShardPlan)]),
    "vstab_offline_fused_plan": (C.c_int, [C.c_long, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.POINTER(FusedPlan)]),
    "vstab_offline_run": (C.c_int, [_vp, C.POINTER(OfflineCfg), C.POINTER(OfflineReport)]),
    "vstab_frame_checksum": (C.c_uint64, [_vp, C.c_int, C.c_int, C.c_size_t]),
    "vstab_offline_prepare": (C.c_int, [_vp, _vp, C.c_long, C.c_int, C.c_long]),
    "vstab_offline_set_timing": (None, [_vp, C.c_int]),
    "vstab_offline_stage_times": (C.c_int, [_vp, _f32p, C.POINTER(C.c_int)]),
    "vstab_launch_count": (C.c_longlong, []),
    "vstab_debug_guard_violations": (C.c_longlong, []),
    "vstab_debug_link_probe": (C.c_int, [C.c_int, _vp, _vp, C.c_size_t, C.c_size_t, C.c_int, C.POINTER(C.c_double)]),
    "vstab_debug_guard_buffers": (C.c_longlong, []),
    "vstab_offline_read_h": (C.c_long, [_vp, _f64p, C.c_size_t]),
    "vstab_offline_stream": (C.c_size_t, [_vp]),
    "vstab_render_frames": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int, _f64p, C.c_int, C.c_int, C.c_int, C.c_double,
                                      _vp, C.c_size_t, C.c_size_t]),
    "vstab_k_ingest": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int, C.c_size_t, C.c_int, _vp, C.POINTER(C.c_uint64)]),
    "vstab_k_pyramid": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int, _vp, _vp, _vp]),
    "vstab_k_gftt": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, _vp, C.POINTER(C.c_int), _vp]),
    "vstab_k_lk": (C.c_int, [C.c_int, _vp, _vp, C.c_int, C.c_int, _vp, C.c_int, _vp, _vp]),
    "vstab_k_fit": (C.c_int, [C.c_int, _vp, _vp, _vp, C.c_int, C.c_double, C.c_int, C.c_int, _f64p, _f64p,
                              C.POINTER(C.c_int)]),
    "vstab_k_warp": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int, C.c_size_t, _f64p, _vp, _vp, C.c_size_t]),
    "vstab_k_featprep": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int, C.c_size_t, C.c_int, _vp]),
    "vstab_k_orb": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int, C.c_double, C.c_int, _vp, _vp, C.POINTER(C.c_int), C.c_int]),
    "vstab_k_hamming": (C.c_int, [C.c_int, _vp, C.c_int, _vp, C.c_int, C.c_float, _vp, _vp, _vp, _vp]),
    "vstab_k_l2match": (C.c_int, [C.c_int, _vp, C.c_int, _vp, C.c_int, _vp, _vp, _vp]),
    "vstab_k_l2match_batch": (C.c_int, [C.c_int, _vp, C.c_int, _vp, C.POINTER(C.c_int), C.c_int, _vp, _vp, C.c_int, C.POINTER(C.c_float)]),
    "vstab_k_sift": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int, C.c_double, _vp, _vp, C.POINTER(C.c_int), C.c_int]),
    "vstab_k_sift_stages": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int, C.c_double, C.c_int, _vp, _vp, C.c_size_t, _vp, C.c_int,
                                      _vp, C.c_int, _vp, _vp, _vp, C.POINTER(C.c_int), C.c_int]),
    "vstab_k_sift_extrema": (C.c_int, [C.c_int, _vp, C.c_size_t, C.c_int, C.c_int, _vp, C.c_int, _vp]),
    "vstab_k_fit_large": (C.c_int, [C.c_int, _vp, _vp, _vp, C.c_int, C.c_double, C.c_int, C.c_int, _f64p, _f64p,
                                    C.POINTER(C.c_int)]),
}

_lib = None


def load_library(path: str | None = None) -> C.CDLL:
    """Load libvstab.so and bind every declared symbol.  Raises if the library is missing:
    there is deliberately no fallback implementation."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise VstabError(f"{p} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                         f"(or `make -C video-stabilization_b200`); there is no CPU fallback")
    lib = C.CDLL(p)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the ABI lost a symbol
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(_vp)


def _check(st: int, handle=None, offline: bool = False):
    if st == OK:
        return
    lib = load_library()
    msg = lib.vstab_offline_last_error(handle) if offline else lib.vstab_last_error(handle)
    msg = msg.decode() if msg else lib.vstab_status_string(st).decode()
    if st in (ERR_INVALID_ARGUMENT, ERR_SIZE_CHANGED):
        raise ValueError(msg)                # std::invalid_argument in the reference
    if st == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if st == ERR_STATE:
        raise AssertionError(msg)            # the reference asserts (stabilizer.cpp:329)
    raise VstabError(msg)


def frame_checksum(img: np.ndarray) -> int:
    """The per-frame output checksum the warp kernel accumulates (csrc/warp.cu, include/vstab.h vstab_frame_checksum):
    rows cut into 12-byte groups (4 pixels, zero-padded) read as three little-endian words,
    sum_y sum_g (y + 1)(g + 1)(w0 + 3 w1 + 5 w2) mod 2^64.  numpy twin of the C function."""
    h, w, _ = img.shape
    wp = (w + 3) // 4 * 4
    row = np.zeros((h, wp * 3), np.uint8)
    row[:, :w * 3] = img.reshape(h, -1)
    wd = row.view("<u4").reshape(h, wp // 4, 3).astype(np.uint64)
    t = wd[..., 0] + np.uint64(3) * wd[..., 1] + np.uint64(5) * wd[..., 2]
    with np.errstate(over="ignore"):
        t = t * (np.arange(h, dtype=np.uint64) + np.uint64(1))[:, None] * (np.arange(wp // 4, dtype=np.uint64) + np.uint64(1))[None, :]
        return int(t.sum(dtype=np.uint64))


CROP_RELEASE = 0.002      # default zoom release per call of set_crop and the front ends' --crop


def crop_zoom(H: np.ndarray, rows: int, cols: int, max_zoom: float) -> float:
    """The zoom about the centre a rows x cols frame warped by H needs to show no border (vstab_crop_zoom), at most
    max_zoom.  Host only."""
    Hc = np.ascontiguousarray(np.asarray(H, np.float64).reshape(9))
    z = float(load_library().vstab_crop_zoom(Hc.ctypes.data_as(_f64p), int(rows), int(cols), float(max_zoom)))
    if z < 0:
        raise ValueError("crop_zoom: rows and cols must be >= 2 and max_zoom in [1, 4]")
    return z


def yuv_layout_packed(fmt: int, rows: int, cols: int):
    """The tight rawvideo layout of a rows x cols NV12 / I420 frame -> (YuvLayout, frame bytes).  Host only."""
    L = YuvLayout()
    n = load_library().vstab_yuv_layout_packed(int(fmt), int(rows), int(cols), C.byref(L))
    if n == 0:
        raise ValueError(f"no 4:2:0 layout for format {fmt} at {rows}x{cols} (formats PIX_NV12 / PIX_I420, even sizes)")
    return L, int(n)


def _yuv_frame_rows(frame: np.ndarray) -> int:
    """rows of a packed 4:2:0 frame array [rows * 3 // 2, cols]"""
    if not isinstance(frame, np.ndarray) or frame.dtype != np.uint8 or frame.ndim != 2 or frame.shape[0] % 3:
        raise ValueError("a packed 4:2:0 frame is a uint8 array [rows * 3 // 2, cols]")
    return frame.shape[0] * 2 // 3


@dataclass
class HomographyParameters:
    s: float = 1.0
    theta: float = 0.0
    k: float = 1.0
    delta: float = 0.0
    t: tuple = (0.0, 0.0)
    v: tuple = (0.0, 0.0)


class Stabilizer:
    """Drop-in for the reference's Stabilizer on the LK + warp path (device-resident state)."""

    def __init__(self, past_frames: int = 15, future_frames: int = 15, working_height: int = 360,
                 device: int = 0):
        self._lib = load_library()
        self._h = _vp()
        _check(self._lib.vstab_create(past_frames, future_frames, working_height, device, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.vstab_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def total_frame_window_size(self) -> int:
        return int(self._lib.vstab_total_frame_window_size(self._h))

    def set_trail(self, enable: bool) -> None:
        """The copyFeathered branch of stabilizeFrame (src/stabilizer.cpp:1303-1307), off by default as in the reference."""
        _check(self._lib.vstab_set_trail(self._h, 1 if enable else 0), self._h)

    def set_partial_lock_fix(self, enable: bool) -> None:
        """TRANSLATION_/ROTATION_LOCK from the accumulated lock (src/stabilizer.cpp:1246-1260 fed as intended; the
        reference returns the identity in these modes, which stays the default)."""
        _check(self._lib.vstab_set_partial_lock_fix(self._h, 1 if enable else 0), self._h)

    def set_crop(self, max_zoom: float, release: float = CROP_RELEASE) -> None:
        """Auto-crop (vstab_set_crop): zoom each output about its centre just enough to hide the border of its warp, at most
        `max_zoom` (1 < max_zoom <= 4; 1.0 turns it off), falling back by at most `release` per call."""
        _check(self._lib.vstab_set_crop(self._h, float(max_zoom), float(release)), self._h)

    def set_stabilization_mode(self, mode: int) -> None:
        _check(self._lib.vstab_set_mode(self._h, int(mode)), self._h)

    def stabilize_frame(self, frame: np.ndarray, out: np.ndarray | None = None) -> np.ndarray:
        if frame.dtype != np.uint8 or frame.ndim != 3 or frame.shape[2] != 3:
            raise ValueError("frame must be HxWx3 uint8 (BGR)")
        if frame.strides[2] != 1 or frame.strides[1] != 3:
            frame = np.ascontiguousarray(frame)
        if out is None:
            out = np.empty((frame.shape[0], frame.shape[1], 3), np.uint8)
        elif (not isinstance(out, np.ndarray) or out.dtype != np.uint8 or out.shape != frame.shape or out.strides[2] != 1
              or out.strides[1] != 3 or out.strides[0] < 3 * frame.shape[1] or not out.flags.writeable):
            # the native call writes rows * cols * 3 bytes at out.strides[0]: anything else would be out of bounds
            raise ValueError("out must be a writeable uint8 array of the frame's shape with packed BGR pixels")
        _check(self._lib.vstab_stabilize_frame(self._h, _ptr(frame), frame.shape[0], frame.shape[1],
                                               frame.strides[0], _ptr(out), out.strides[0]), self._h)
        return out

    def stabilize_frame_yuv(self, frame: np.ndarray, fmt: int, out: np.ndarray | None = None,
                            out_fmt: int | None = None) -> np.ndarray:
        """stabilize_frame on a packed NV12 / I420 frame [rows * 3 // 2, cols] (ffmpeg rawvideo); returns the output as a
        packed frame of `out_fmt` (default: `fmt`).  Equals to_yuv(stabilize_frame(from_yuv(frame))) call by call."""
        rows = _yuv_frame_rows(frame)
        cols = frame.shape[1]
        out_fmt = fmt if out_fmt is None else out_fmt
        frame = np.ascontiguousarray(frame)
        if out is None:
            out = np.empty_like(frame)
        elif (not isinstance(out, np.ndarray) or out.shape != frame.shape or out.dtype != np.uint8 or not out.flags.c_contiguous
              or not out.flags.writeable):
            raise ValueError("out must be a writeable C-contiguous uint8 array of the frame's shape")
        # the library checks formats and sizes (odd sizes have no packed layout: pass one it rejects with its own message)
        lin, lout = (YuvLayout.make(f, [0, 0, 0], [cols] * 3) for f in (fmt, out_fmt))
        if rows > 0 and cols > 0 and rows % 2 == 0 and cols % 2 == 0 and fmt in (PIX_NV12, PIX_I420) and out_fmt in (PIX_NV12, PIX_I420):
            lin, lout = yuv_layout_packed(fmt, rows, cols)[0], yuv_layout_packed(out_fmt, rows, cols)[0]
        _check(self._lib.vstab_stabilize_frame_yuv(self._h, _ptr(frame), C.byref(lin), rows, cols, _ptr(out), C.byref(lout)), self._h)
        return out

    def stabilize_frame_yuv_ptr(self, src_ptr: int, layout: YuvLayout, rows: int, cols: int, dst_ptr: int,
                                out_layout: YuvLayout, device: bool = False) -> None:
        """YUV call on raw frame base pointers (host, or device with device=True: asynchronous, see synchronize())."""
        fn = self._lib.vstab_stabilize_frame_yuv_device if device else self._lib.vstab_stabilize_frame_yuv
        _check(fn(self._h, _vp(src_ptr), C.byref(layout), rows, cols, _vp(dst_ptr), C.byref(out_layout)), self._h)

    def stabilize_frame_ptr(self, src_ptr: int, rows: int, cols: int, step: int, dst_ptr: int, dst_step: int,
                            device: bool = False) -> None:
        fn = self._lib.vstab_stabilize_frame_device if device else self._lib.vstab_stabilize_frame
        _check(fn(self._h, _vp(src_ptr), rows, cols, step, _vp(dst_ptr), dst_step), self._h)

    def synchronize(self) -> None:
        _check(self._lib.vstab_synchronize(self._h), self._h)

    # ---- parity taps ------------------------------------------------------------------
    def working_size(self):
        return self._lib.vstab_working_width(self._h), self._lib.vstab_working_height(self._h)

    def presentation_index(self) -> int:
        return int(self._lib.vstab_presentation_index(self._h))

    def tap(self, which: int) -> np.ndarray:
        ww, wh = self.working_size()
        spec = {
            TAP_GRAY: (np.uint8, ww * wh), TAP_PYR1: (np.uint8, ww * wh), TAP_PYR2: (np.uint8, ww * wh),
            TAP_PYR3: (np.uint8, ww * wh), TAP_PREV_PTS: (np.float32, 2600), TAP_LK_PTS: (np.float32, 2600),
            TAP_LK_STATUS: (np.uint8, 1300), TAP_NEW_PTS: (np.float32, 2600), TAP_T: (np.float64, 9),
            TAP_M: (np.float64, 6), TAP_H_STABILIZE: (np.float64, 9), TAP_H_SCALED: (np.float64, 9),
            TAP_BORDER: (np.uint8, 3), TAP_EIG: (np.float32, ww * wh), TAP_INLIERS: (np.int32, 2),
            TAP_CHANNEL_SUMS: (np.uint64, 3), TAP_LOCK_H: (np.float64, 9), TAP_ORB_COUNTS: (np.int32, 5),
            TAP_FEAT_GRAY: (np.uint8, ww * wh),
        }[which]
        buf = np.zeros(spec[1], spec[0])
        n = self._lib.vstab_read_tap(self._h, which, _ptr(buf), buf.nbytes)
        if n < 0:
            raise VstabError(f"tap {which} failed ({n})")
        if which in (TAP_PREV_PTS, TAP_LK_PTS, TAP_NEW_PTS):
            return buf[:2 * n].reshape(-1, 2)
        if which in (TAP_GRAY, TAP_EIG, TAP_FEAT_GRAY):
            return buf[:n].reshape(wh, ww)
        if which in (TAP_PYR1, TAP_PYR2, TAP_PYR3):
            l = which - TAP_PYR1 + 1
            w_, h_ = ww, wh
            for _ in range(l):
                w_, h_ = (w_ + 1) // 2, (h_ + 1) // 2
            return buf[:n].reshape(h_, w_)
        if which in (TAP_T, TAP_H_STABILIZE, TAP_H_SCALED, TAP_LOCK_H):
            return buf[:n].reshape(3, 3)
        if which == TAP_M:
            return buf[:n].reshape(2, 3)
        return buf[:n]

    # ---- static helpers ----------------------------------------------------------------
    @staticmethod
    def decompose_homography(H: np.ndarray, center=(0.0, 0.0)):
        H = np.asarray(H)
        if H.shape != (3, 3) or H.dtype != np.float64:
            raise ValueError("Error: Input homography matrix must be a non-empty 3x3 CV_64F matrix.")
        Hc = np.ascontiguousarray(H)
        hp = HParams()
        r = load_library().vstab_decompose_homography(Hc.ctypes.data_as(_f64p), center[0], center[1], C.byref(hp))
        if r < 0:
            raise ValueError("bad argument")
        if r == 0:
            return None
        return HomographyParameters(hp.s, hp.theta, hp.k, hp.delta, (hp.t[0], hp.t[1]), (hp.v[0], hp.v[1]))

    @staticmethod
    def compose_homography(p: HomographyParameters, center=(0.0, 0.0)) -> np.ndarray:
        hp = HParams(p.s, p.theta, p.k, p.delta, (C.c_double * 2)(*p.t), (C.c_double * 2)(*p.v))
        H = np.zeros((3, 3))
        load_library().vstab_compose_homography(C.byref(hp), center[0], center[1], H.ctypes.data_as(_f64p))
        return H


# ---- single-kernel entry points (host arrays) ----------------------------------------------
def k_ingest(bgr: np.ndarray, working_height: int, device: int = 0):
    lib = load_library()
    rows, cols = bgr.shape[:2]
    s = float(working_height) / rows
    ww = int(cols * s)
    gray = np.empty((working_height, ww), np.uint8)
    sums = (C.c_uint64 * 3)()
    bgr = np.ascontiguousarray(bgr)
    _check(lib.vstab_k_ingest(device, _ptr(bgr), rows, cols, bgr.strides[0], working_height, _ptr(gray), sums))
    return gray, np.array(list(sums), dtype=np.uint64)


def k_pyramid(gray: np.ndarray, device: int = 0):
    lib = load_library()
    h, w = gray.shape
    outs = []
    for _ in range(3):
        w, h = (w + 1) // 2, (h + 1) // 2
        outs.append(np.empty((h, w), np.uint8))
    gray = np.ascontiguousarray(gray)
    _check(lib.vstab_k_pyramid(device, _ptr(gray), gray.shape[0], gray.shape[1], *[_ptr(o) for o in outs]))
    return outs


def k_gftt(gray: np.ndarray, max_corners=1300, quality=0.01, min_distance=5, want_eig=False, device: int = 0):
    lib = load_library()
    gray = np.ascontiguousarray(gray)
    pts = np.zeros((1300, 2), np.float32)
    n = C.c_int(0)
    eig = np.zeros(gray.shape, np.float32) if want_eig else None
    _check(lib.vstab_k_gftt(device, _ptr(gray), gray.shape[0], gray.shape[1], max_corners, quality, min_distance,
                            _ptr(pts), C.byref(n), _ptr(eig) if want_eig else None))
    return (pts[:n.value].copy(), eig) if want_eig else pts[:n.value].copy()


def k_lk(prev: np.ndarray, nxt: np.ndarray, pts: np.ndarray, device: int = 0):
    lib = load_library()
    prev = np.ascontiguousarray(prev)
    nxt = np.ascontiguousarray(nxt)
    pts = np.ascontiguousarray(pts, np.float32)
    n = len(pts)
    out = np.zeros((n, 2), np.float32)
    st = np.zeros(n, np.uint8)
    _check(lib.vstab_k_lk(device, _ptr(prev), _ptr(nxt), prev.shape[0], prev.shape[1], _ptr(pts), n, _ptr(out), _ptr(st)))
    return out, st


def k_fit(prev_pts, next_pts, status, work_w, work_h, thresh=3.0, device: int = 0):
    lib = load_library()
    a = np.ascontiguousarray(prev_pts, np.float32)
    b = np.ascontiguousarray(next_pts, np.float32)
    s = np.ascontiguousarray(status, np.uint8)
    M = np.zeros((2, 3))
    T = np.zeros((3, 3))
    cnt = (C.c_int * 2)()
    _check(lib.vstab_k_fit(device, _ptr(a), _ptr(b), _ptr(s), len(a), thresh, work_w, work_h,
                           M.ctypes.data_as(_f64p), T.ctypes.data_as(_f64p), cnt))
    return M, T, (cnt[0], cnt[1])


def k_fit_large(ref_pts, cur_pts, status, work_w, work_h, thresh=5.0, device: int = 0):
    """k_fit's estimator instantiated for up to 4096 pairs (the ORB / SIFT registration fit)."""
    lib = load_library()
    a = np.ascontiguousarray(ref_pts, np.float32)
    b = np.ascontiguousarray(cur_pts, np.float32)
    s = np.ascontiguousarray(status, np.uint8)
    M = np.zeros((2, 3))
    T = np.zeros((3, 3))
    cnt = (C.c_int * 2)()
    _check(lib.vstab_k_fit_large(device, _ptr(a), _ptr(b), _ptr(s), len(a), thresh, work_w, work_h,
                                 M.ctypes.data_as(_f64p), T.ctypes.data_as(_f64p), cnt))
    return M, T, (cnt[0], cnt[1])


def k_warp(bgr: np.ndarray, H: np.ndarray, border, device: int = 0):
    lib = load_library()
    bgr = np.ascontiguousarray(bgr)
    H = np.ascontiguousarray(H, np.float64)
    b = np.array(list(border)[:3], np.uint8)
    out = np.empty_like(bgr)
    _check(lib.vstab_k_warp(device, _ptr(bgr), bgr.shape[0], bgr.shape[1], bgr.strides[0], H.ctypes.data_as(_f64p),
                            _ptr(b), _ptr(out), out.strides[0]))
    return out


def k_yuv_to_bgr(yuv: np.ndarray, layout, rows: int | None = None, cols: int | None = None, device: int = 0) -> np.ndarray:
    """cvtColor(YUV2BGR_NV12 / _I420) on the GPU (K15).  `layout`: PIX_NV12 / PIX_I420 for a packed frame
    [rows * 3 // 2, cols], or a YuvLayout of the frame whose base is yuv's first byte (then rows, cols are required)."""
    lib = load_library()
    yuv = np.ascontiguousarray(yuv)
    if not isinstance(layout, YuvLayout):
        rows, cols = _yuv_frame_rows(yuv), yuv.shape[1]
        layout = yuv_layout_packed(layout, rows, cols)[0]
    out = np.empty((rows, cols, 3), np.uint8)
    _check(lib.vstab_k_yuv_to_bgr(device, _ptr(yuv), C.byref(layout), rows, cols, _ptr(out), out.strides[0]))
    return out


def k_bgr_to_yuv(bgr: np.ndarray, layout, out: np.ndarray | None = None, device: int = 0) -> np.ndarray:
    """cvtColor(BGR2YUV_I420) on the GPU (K15; NV12 = its chroma interleaved U,V).  `layout`: PIX_NV12 / PIX_I420 returns a
    packed frame [rows * 3 // 2, cols]; a YuvLayout writes its planes into `out` (a C-contiguous buffer holding the frame)."""
    lib = load_library()
    bgr = np.ascontiguousarray(bgr)
    rows, cols = bgr.shape[:2]
    if not isinstance(layout, YuvLayout):
        layout = yuv_layout_packed(layout, rows, cols)[0]
        out = np.zeros((rows * 3 // 2, cols), np.uint8)
    elif out is None or not out.flags.c_contiguous or not out.flags.writeable:
        raise ValueError("a YuvLayout needs a writeable C-contiguous `out` buffer")
    _check(lib.vstab_k_bgr_to_yuv(device, _ptr(bgr), rows, cols, bgr.strides[0], _ptr(out), C.byref(layout)))
    return out


def k_copy_feathered(fg: np.ndarray, bg: np.ndarray, H: np.ndarray, device: int = 0) -> np.ndarray:
    """Stabilizer::copyFeathered (src/stabilizer.cpp:1051-1155) on the GPU."""
    lib = load_library()
    fg = np.ascontiguousarray(fg)
    bg = np.ascontiguousarray(bg)
    if fg.shape != bg.shape:
        raise ValueError("Stabilizer: copyFeathered: foreground and background_image must have the same size")
    H = np.ascontiguousarray(H, np.float64)
    out = np.empty_like(fg)
    _check(lib.vstab_k_copy_feathered(device, _ptr(fg), _ptr(bg), fg.shape[0], fg.shape[1], fg.strides[0],
                                      H.ctypes.data_as(_f64p), _ptr(out), out.strides[0]))
    return out


def k_featprep(bgr: np.ndarray, working_height: int, device: int = 0) -> np.ndarray:
    """ORB/SIFT preprocessing chain of the reference (src/stabilizer.cpp:448-477) on the GPU."""
    lib = load_library()
    rows, cols = bgr.shape[:2]
    ww = int(cols * (float(working_height) / rows))
    out = np.empty((working_height, ww), np.uint8)
    bgr = np.ascontiguousarray(bgr)
    _check(lib.vstab_k_featprep(device, _ptr(bgr), rows, cols, bgr.strides[0], working_height, _ptr(out)))
    return out


def k_orb(gray: np.ndarray, size_ratio: float = 0.0, reference_order: bool = False, device: int = 0):
    """ORB(2500, 1.2, 12, 31, 0, 2, FAST_SCORE, 31, 20).detectAndCompute -> (kps [n,6], desc [n,32])."""
    lib = load_library()
    gray = np.ascontiguousarray(gray)
    kps = np.zeros((4096, 6), np.float32)
    desc = np.zeros((4096, 32), np.uint8)
    n = C.c_int(0)
    _check(lib.vstab_k_orb(device, _ptr(gray), gray.shape[0], gray.shape[1], float(size_ratio), int(reference_order), _ptr(kps), _ptr(desc),
                           C.byref(n), 4096))
    return kps[:n.value].copy(), desc[:n.value].copy()


def k_hamming(ref: np.ndarray, cur: np.ndarray, ratio: float = 0.6, device: int = 0):
    """BFMatcher(NORM_HAMMING).knnMatch(ref, cur, 2) + ratio test -> (best_idx, best_d, second_d, good)."""
    lib = load_library()
    ref = np.ascontiguousarray(ref, np.uint8)
    cur = np.ascontiguousarray(cur, np.uint8)
    n = len(ref)
    bi = np.zeros(n, np.int32); bd = np.zeros(n, np.int32); sd = np.zeros(n, np.int32); good = np.zeros(n, np.uint8)
    _check(lib.vstab_k_hamming(device, _ptr(ref), n, _ptr(cur), len(cur), ratio, _ptr(bi), _ptr(bd), _ptr(sd), _ptr(good)))
    return bi, bd, sd, good


def k_l2match(ref: np.ndarray, cur: np.ndarray, device: int = 0):
    """BFMatcher(NORM_L2).match(ref, cur) on tcgen05 + the reference's distance filter
    -> (best_idx, best_d2 (exact squared distance), good).  Descriptors: integer valued [n,128]."""
    lib = load_library()
    ref8 = np.ascontiguousarray(ref).astype(np.uint8)
    cur8 = np.ascontiguousarray(cur).astype(np.uint8)
    if not (np.array_equal(ref8, ref) and np.array_equal(cur8, cur)):
        raise ValueError("descriptors must be integers in 0..255")
    n = len(ref8)
    bi = np.zeros(n, np.int32); bd = np.zeros(n, np.int32); good = np.zeros(n, np.uint8)
    _check(lib.vstab_k_l2match(device, _ptr(ref8), n, _ptr(cur8), len(cur8), _ptr(bi), _ptr(bd), _ptr(good)))
    return bi, bd, good


def k_l2match_batch(ref: np.ndarray, curs, reps: int = 1, device: int = 0):
    """Nearest neighbours of every row of `ref` in each of the descriptor sets `curs` (one launch for the whole batch)
    -> (best_idx [n, nref], best_d2 [n, nref], ms per launch)."""
    lib = load_library()
    ref8 = np.ascontiguousarray(ref, np.uint8)
    cat = np.ascontiguousarray(np.concatenate([np.asarray(c, np.uint8) for c in curs], 0))
    ncur = (C.c_int * len(curs))(*[len(c) for c in curs])
    bi = np.zeros((len(curs), len(ref8)), np.int32); bd = np.zeros((len(curs), len(ref8)), np.int32)
    ms = C.c_float(0)
    _check(lib.vstab_k_l2match_batch(device, _ptr(ref8), len(ref8), _ptr(cat), ncur, len(curs), _ptr(bi), _ptr(bd), reps, C.byref(ms)))
    return bi, bd, float(ms.value)


def k_sift(gray: np.ndarray, size_ratio: float = 0.0, device: int = 0):
    """SIFT(2500, 3, 0.04, 5, 1.2).detectAndCompute -> (kps [n,6] {x,y,size,angle,response,octave}, desc u8 [n,128])."""
    lib = load_library()
    gray = np.ascontiguousarray(gray)
    kps = np.zeros((4096, 6), np.float32)
    desc = np.zeros((4096, 128), np.uint8)
    n = C.c_int(0)
    _check(lib.vstab_k_sift(device, _ptr(gray), gray.shape[0], gray.shape[1], float(size_ratio), _ptr(kps), _ptr(desc),
                            C.byref(n), 4096))
    return kps[:n.value].copy(), desc[:n.value].copy()


SIFT_KP_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"), ("octave", "<i4")])


@dataclass
class SiftStages:
    """What vstab_k_sift_stages reads back: `pyr[o]` float32 [6, h, w] per octave, `cand` uint64 DoG extrema
    (octave << 56 | layer << 48 | row << 24 | col), `kps_pre` SIFT_KP_DTYPE records before duplicate removal and
    selection, the raw counters and capacities, `n_sel` the keypoints selected (the output keeps the first 4096), and the
    final keypoints / descriptors as k_sift returns them."""
    pyr: list
    cand: np.ndarray
    n_cand: int
    cand_cap: int
    kps_pre: np.ndarray
    n_kp: int
    kp_cap: int
    n_sel: int
    kps: np.ndarray
    desc: np.ndarray


def k_sift_stages(gray: np.ndarray, size_ratio: float = 0.0, calls: int = 1, device: int = 0) -> SiftStages:
    """vstab_k_sift_stages: one plan, `calls` runs (graph capture from the second, replay from the third), every stage
    of the last run."""
    lib = load_library()
    gray = np.ascontiguousarray(gray, np.uint8)
    rows, cols = gray.shape
    geom = np.zeros(37, np.int32)
    # bounds: the octaves of the 2x base image hold at most 4/3 of its pixels, 6 Gaussians each, each octave padded
    # to 64 floats; candidates at most the capacity the plan gives them (base pixels / 16 + 65536, rounded up to 256)
    pyr = np.zeros(6 * (4 * rows * cols * 4 // 3) + 64 * 12, np.float32)
    cand_max = 4 * rows * cols // 16 + 65536 + 256
    cand = np.zeros(cand_max, np.uint64)
    kp_max = 1 << 18
    pre = np.zeros(kp_max, SIFT_KP_DTYPE)
    counts = np.zeros(5, np.int32)
    kps = np.zeros((4096, 6), np.float32)
    desc = np.zeros((4096, 128), np.uint8)
    n = C.c_int(0)
    _check(lib.vstab_k_sift_stages(device, _ptr(gray), rows, cols, float(size_ratio), int(calls), _ptr(geom), _ptr(pyr),
                                   pyr.size, _ptr(cand), cand_max, _ptr(pre), kp_max, _ptr(counts), _ptr(kps), _ptr(desc),
                                   C.byref(n), 4096))
    levels = []
    for o in range(int(geom[0])):
        w, h, off = int(geom[1 + o]), int(geom[13 + o]), int(geom[25 + o])
        levels.append(pyr[off:off + 6 * w * h].reshape(6, h, w).copy())
    n_cand, n_kp = int(counts[0]), int(counts[2])
    return SiftStages(levels, cand[:min(n_cand, int(counts[1]), cand_max)].copy(), n_cand, int(counts[1]),
                      pre[:min(n_kp, int(counts[3]), kp_max)].copy(), n_kp, int(counts[3]), int(counts[4]),
                      kps[:n.value].copy(), desc[:n.value].copy())


def k_sift_extrema(pyr, rows: int, cols: int, device: int = 0):
    """The DoG extrema pass alone on a caller-made Gaussian pyramid (list over octaves of float32 [6, h, w] in the
    geometry of a rows x cols input) -> (candidate words uint64, found, capacity)."""
    lib = load_library()
    flat = np.ascontiguousarray(np.concatenate([np.asarray(g, np.float32).ravel() for g in pyr]))
    cand_max = 4 * rows * cols // 16 + 65536 + 256
    cand = np.zeros(cand_max, np.uint64)
    counts = np.zeros(2, np.int32)
    _check(lib.vstab_k_sift_extrema(device, _ptr(flat), flat.size, rows, cols, _ptr(cand), cand_max, _ptr(counts)))
    return cand[:min(int(counts[0]), int(counts[1]), cand_max)].copy(), int(counts[0]), int(counts[1])
