"""YUV 4:2:0 frames without a GPU: the numpy restatements of OpenCV's conversions (tests/yuv_ref.py, what K15 implements)
are bit-identical to cv2, the packed rawvideo layouts of the C ABI, its argument checks, and the --pix-fmt flags of the
file front end (examples/vstab_file.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import __graft_entry__ as entry
import vstab_b200 as vs
from yuv_ref import I420, NV12, bgr_to_yuv420, join_planes, split_planes, yuv420_to_bgr

cv2 = pytest.importorskip("cv2")

SIZES = [(1080, 1920), (2160, 3840), (360, 640), (250, 334), (126, 202), (14, 18), (12, 12)]


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(vs.LIB_PATH):
        entry.build()
    return vs.load_library()


def _cv_to_bgr(frame, fmt):
    return cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12 if fmt == NV12 else cv2.COLOR_YUV2BGR_I420)


def _cv_to_yuv(bgr, fmt):
    i420 = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)
    return i420 if fmt == I420 else join_planes(*split_planes(i420, I420), NV12)


@pytest.mark.parametrize("rows,cols", SIZES)
def test_restatements_equal_cv2_on_random_frames(rows, cols):
    """Odd half widths (334 x 250, 202 x 126) included: the chroma planes have an odd number of columns."""
    rng = np.random.default_rng(rows * 7 + cols)
    yuv = rng.integers(0, 256, (rows * 3 // 2, cols), dtype=np.uint8)
    bgr = rng.integers(0, 256, (rows, cols, 3), dtype=np.uint8)
    for fmt in (NV12, I420):
        assert np.array_equal(yuv420_to_bgr(yuv, fmt), _cv_to_bgr(yuv, fmt)), fmt
        assert np.array_equal(bgr_to_yuv420(bgr, fmt), _cv_to_yuv(bgr, fmt)), fmt
    # NV12 and I420 of the same planes decode to the same picture
    Y, U, V = split_planes(yuv, I420)
    assert np.array_equal(yuv420_to_bgr(join_planes(Y, U, V, NV12), NV12), yuv420_to_bgr(yuv, I420))


@pytest.mark.parametrize("value", [0, 255, "low"])
def test_restatements_equal_cv2_at_the_ends_of_the_range(value):
    """all-0, all-255 and Y < 16 (the luma term clamps at 0) inputs"""
    rows, cols = 24, 34
    if value == "low":
        yuv = np.random.default_rng(1).integers(0, 16, (rows * 3 // 2, cols), dtype=np.uint8)
        yuv[rows:] = np.random.default_rng(2).integers(0, 256, (rows // 2, cols), dtype=np.uint8)
    else:
        yuv = np.full((rows * 3 // 2, cols), value, np.uint8)
    bgr = np.full((rows, cols, 3), 0 if value == "low" else value, np.uint8)
    for fmt in (NV12, I420):
        assert np.array_equal(yuv420_to_bgr(yuv, fmt), _cv_to_bgr(yuv, fmt))
        assert np.array_equal(bgr_to_yuv420(bgr, fmt), _cv_to_yuv(bgr, fmt))


@pytest.mark.parametrize("rows,cols", [(1080, 1920), (250, 334), (12, 12)])
def test_packed_layouts(lib, rows, cols):
    """vstab_yuv_layout_packed: ffmpeg's rawvideo planes (nv12: Y then U,V pairs; yuv420p: Y, U, V)"""
    L, n = vs.yuv_layout_packed(vs.PIX_NV12, rows, cols)
    assert n == rows * cols * 3 // 2 and L.format == vs.PIX_NV12
    assert list(L.offset)[:2] == [0, rows * cols] and list(L.step)[:2] == [cols, cols]
    L, n = vs.yuv_layout_packed(vs.PIX_I420, rows, cols)
    assert n == rows * cols * 3 // 2 and L.format == vs.PIX_I420
    assert list(L.offset) == [0, rows * cols, rows * cols + rows * cols // 4] and list(L.step) == [cols, cols // 2, cols // 2]


def test_packed_layout_rejects_odd_sizes_and_unknown_formats(lib):
    L = vs.YuvLayout()
    for fmt, rows, cols in [(vs.PIX_NV12, 1080, 1919), (vs.PIX_I420, 1081, 1920), (0, 1080, 1920), (3, 1080, 1920),
                            (vs.PIX_NV12, 0, 0), (vs.PIX_I420, -2, 4)]:
        assert lib.vstab_yuv_layout_packed(fmt, rows, cols, C.byref(L)) == 0, (fmt, rows, cols)
        with pytest.raises(ValueError):
            vs.yuv_layout_packed(fmt, rows, cols)
    assert lib.vstab_yuv_layout_packed(vs.PIX_NV12, 4, 4, None) == 0


def test_abi_argument_checks_before_any_device_work(lib):
    """NULL instances / layouts, unknown formats, odd sizes and short steps are argument errors, checked on the host."""
    L, _ = vs.yuv_layout_packed(vs.PIX_NV12, 64, 64)
    buf = np.zeros(64 * 96, np.uint8)
    p = buf.ctypes.data_as(C.c_void_p)
    assert lib.vstab_stabilize_frame_yuv(None, p, C.byref(L), 64, 64, p, C.byref(L)) == vs.ERR_INVALID_ARGUMENT
    assert lib.vstab_stabilize_frame_yuv_device(None, p, C.byref(L), 64, 64, p, C.byref(L)) == vs.ERR_INVALID_ARGUMENT
    assert lib.vstab_offline_set_yuv(None, None, None) == vs.ERR_INVALID_ARGUMENT
    bgr = np.zeros((64, 64, 3), np.uint8)
    bad = [vs.YuvLayout.make(0, [0, 4096], [64, 64]),                    # unknown format
           vs.YuvLayout.make(vs.PIX_NV12, [0, 4096], [63, 64]),          # Y step below 64 bytes
           vs.YuvLayout.make(vs.PIX_I420, [0, 4096, 5120], [64, 31, 32])]  # U step below 32 bytes
    for b in bad:
        assert lib.vstab_k_yuv_to_bgr(0, p, C.byref(b), 64, 64, bgr.ctypes.data_as(C.c_void_p), 192) == vs.ERR_INVALID_ARGUMENT
        assert lib.vstab_k_bgr_to_yuv(0, bgr.ctypes.data_as(C.c_void_p), 64, 64, 192, p, C.byref(b)) == vs.ERR_INVALID_ARGUMENT
    assert lib.vstab_k_yuv_to_bgr(0, p, None, 64, 64, bgr.ctypes.data_as(C.c_void_p), 192) == vs.ERR_INVALID_ARGUMENT
    assert lib.vstab_k_yuv_to_bgr(0, p, C.byref(L), 63, 64, bgr.ctypes.data_as(C.c_void_p), 192) == vs.ERR_INVALID_ARGUMENT
    with pytest.raises(ValueError):
        vs.k_yuv_to_bgr(np.zeros((15, 9), np.uint8), vs.PIX_I420)      # 10 x 9: odd width
    with pytest.raises(ValueError):
        vs.k_yuv_to_bgr(np.zeros((7, 10), np.uint8), vs.PIX_NV12)      # not [rows * 3 // 2, cols]


def _front_end():
    exe = os.path.join(os.path.dirname(os.path.dirname(vs.LIB_PATH)), "bin", "vstab_file")
    assert os.path.exists(exe), "video-stabilization_b200/bin/vstab_file is built by make (__graft_entry__.build())"
    return exe


def test_file_front_end_pix_fmt_usage_and_argument_errors(tmp_path, lib):
    """--pix-fmt / --out-pix-fmt take ffmpeg's names; an odd width or height with a 4:2:0 format, a BGR / 4:2:0 mix and
    --side-by-side with 4:2:0 frames are usage errors (exit status 1) before any device is used."""
    exe = _front_end()
    clip = tmp_path / "c.yuv"
    clip.write_bytes(bytes(64 * 48 * 3))
    base = [exe, "--file", str(clip), "--out", str(tmp_path / "o.yuv")]
    for extra in (["--width", "63", "--height", "48", "--pix-fmt", "nv12"],
                  ["--width", "64", "--height", "47", "--pix-fmt", "yuv420p"],
                  ["--width", "64", "--height", "48", "--pix-fmt", "rgb24"],
                  ["--width", "64", "--height", "48", "--pix-fmt", "nv12", "--out-pix-fmt", "bgr24"],
                  ["--width", "64", "--height", "48", "--out-pix-fmt", "nv12"],
                  ["--width", "64", "--height", "48", "--pix-fmt", "nv12", "--side-by-side"],
                  ["--width", "64", "--height", "48", "--pix-fmt"]):
        r = subprocess.run(base + extra, capture_output=True, text=True)
        assert r.returncode == 1, (extra, r.returncode, r.stderr)
    r = subprocess.run([exe, "--help"], capture_output=True, text=True)
    assert "--pix-fmt bgr24|nv12|yuv420p" in r.stderr
    # a valid 4:2:0 command reaches the constructor's checks like a BGR one (workingHeight <= 90: exit 1, no device)
    r = subprocess.run(base + ["--width", "64", "--height", "48", "--pix-fmt", "nv12", "--working-height", "90"],
                       capture_output=True, text=True)
    assert r.returncode == 1 and "workingHeight" in r.stderr
