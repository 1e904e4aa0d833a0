"""numpy restatements of OpenCV's 4:2:0 conversions (cv::cvtColor, BT.601 limited range, 20-bit fixed point) that the K15
kernels (video-stabilization_b200/csrc/yuv.cu) implement, pinned against cv2 in tests/test_yuv.py.  Frames are packed
rawvideo arrays [rows * 3 // 2, cols]: NV12 = Y plane + one interleaved U,V plane, I420 = Y, U, V planes."""
import numpy as np

NV12, I420 = 1, 2            # vstab_pixel_format
_S, _HALF = 20, 1 << 19


def split_planes(frame, fmt):
    """(Y [rows, cols], U [rows/2, cols/2], V [rows/2, cols/2]) of a packed 4:2:0 frame"""
    rows, cols = frame.shape[0] * 2 // 3, frame.shape[1]
    Y = frame[:rows]
    c = frame[rows:].reshape(-1)
    if fmt == NV12:
        uv = c.reshape(rows // 2, cols // 2, 2)
        return Y, uv[..., 0], uv[..., 1]
    q = (rows // 2) * (cols // 2)
    return Y, c[:q].reshape(rows // 2, cols // 2), c[q:].reshape(rows // 2, cols // 2)


def join_planes(Y, U, V, fmt):
    rows, cols = Y.shape
    c = np.stack([U, V], -1).reshape(-1) if fmt == NV12 else np.concatenate([U.reshape(-1), V.reshape(-1)])
    return np.concatenate([Y.reshape(-1), c]).reshape(rows * 3 // 2, cols)


def yuv420_to_bgr(frame, fmt):
    """cvtColor(COLOR_YUV2BGR_NV12 / COLOR_YUV2BGR_I420): the chroma sample of a 2x2 block serves its four pixels"""
    Y, U, V = split_planes(frame, fmt)
    up = lambda p: np.repeat(np.repeat(p.astype(np.int64) - 128, 2, 0), 2, 1)
    u, v = up(U), up(V)
    y = np.maximum(Y.astype(np.int64) - 16, 0) * 1220542
    B = (y + 2116026 * u + _HALF) >> _S
    G = (y - 852492 * v - 409993 * u + _HALF) >> _S
    R = (y + 1673527 * v + _HALF) >> _S
    return np.clip(np.stack([B, G, R], -1), 0, 255).astype(np.uint8)


def bgr_to_yuv420(bgr, fmt):
    """cvtColor(COLOR_BGR2YUV_I420) (NV12: its chroma interleaved U,V): luma of every pixel, chroma of the top-left pixel of
    each 2x2 block (no averaging)"""
    b, g, r = (bgr[..., i].astype(np.int64) for i in range(3))
    Y = (269484 * r + 528482 * g + 102760 * b + _HALF + (16 << _S)) >> _S
    tl = (slice(None, None, 2), slice(None, None, 2))
    U = (-155188 * r[tl] - 305135 * g[tl] + 460324 * b[tl] + _HALF + (128 << _S)) >> _S
    V = (460324 * r[tl] - 385875 * g[tl] - 74448 * b[tl] + _HALF + (128 << _S)) >> _S
    return join_planes(Y.astype(np.uint8), U.astype(np.uint8), V.astype(np.uint8), fmt)
