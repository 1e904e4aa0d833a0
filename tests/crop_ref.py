"""Plain-Python restatement of auto-crop (include/vstab.h vstab_set_crop; csrc/homography.cuh crop_need / crop_apply and
csrc/crop.cu).  Scalar Python floats in the kernels' operation order: crop.cu is built without FMA contraction, so for the
same inputs the device results carry these bits."""
import math

import numpy as np


def crop_r(max_zoom: float, release: float) -> int:
    """R: the number of calls a need stays in the zoom of later calls."""
    return int(math.ceil((max_zoom - 1.0) / release))


def need(H, rows: int, cols: int, max_zoom: float) -> float:
    """The zoom about the centre that keeps the warp by H from showing any point outside the pixel-centre rectangle."""
    h = [float(v) for v in np.asarray(H, np.float64).reshape(9)]
    if not all(math.isfinite(v) for v in h):
        return max_zoom
    xs = [0.0, cols - 1.0, cols - 1.0, 0.0]
    ys = [0.0, 0.0, rows - 1.0, rows - 1.0]
    qx, qy = [0.0] * 4, [0.0] * 4
    for k in range(4):
        w = h[6] * xs[k] + h[7] * ys[k] + h[8]
        if not w > 0.0:
            return max_zoom
        qx[k] = (h[0] * xs[k] + h[1] * ys[k] + h[2]) / w
        qy[k] = (h[3] * xs[k] + h[4] * ys[k] + h[5]) / w
    area2 = 0.0
    for k in range(4):
        area2 = area2 + (qx[k] * qy[(k + 1) & 3] - qx[(k + 1) & 3] * qy[k])
    sg = 1.0 if area2 > 0.0 else -1.0
    cx, cy = (cols - 1.0) * 0.5, (rows - 1.0) * 0.5
    t = 1.0
    for k in range(4):
        ex, ey = qx[(k + 1) & 3] - qx[k], qy[(k + 1) & 3] - qy[k]
        s0 = sg * (ex * (cy - qy[k]) - ey * (cx - qx[k]))
        if not s0 > 0.0:
            return max_zoom
        for j in range(4):
            s1 = sg * (ex * (ys[j] - cy) - ey * (xs[j] - cx))
            if s1 < 0.0:
                b = s0 / -s1
                if b < t:
                    t = b
    z = 1.0 / t
    return 1.0 if z < 1.0 else (max_zoom if z > max_zoom else z)


def zoom_at(needs, base: int, c: int, R: int, release: float, max_zoom: float) -> float:
    """z_c from the needs of calls [max(0, c-R), c]; needs[j - base] is n_j."""
    m = 1.0
    for j in range(max(0, c - R), c + 1):
        m = max(m, needs[j - base] - float(c - j) * release)
    return max_zoom if m > max_zoom else m


def schedule(needs, first: int, n: int, R: int, release: float, max_zoom: float, base: int = 0):
    """z_c for calls [first, first + n) given the needs of calls [base, first + n) (base <= max(0, first - R))."""
    return [zoom_at(needs, base, c, R, release, max_zoom) for c in range(first, first + n)]


def matmul3(A, B):
    C = [0.0] * 9
    for i in range(3):
        for j in range(3):
            s = A[i * 3 + 0] * B[0 * 3 + j]
            s = s + A[i * 3 + 1] * B[1 * 3 + j]
            s = s + A[i * 3 + 2] * B[2 * 3 + j]
            C[i * 3 + j] = s
    return C


def apply(z: float, H, rows: int, cols: int) -> np.ndarray:
    """Hc = Z(z) * H"""
    cx, cy = (cols - 1.0) * 0.5, (rows - 1.0) * 0.5
    Z = [z, 0.0, (1.0 - z) * cx, 0.0, z, (1.0 - z) * cy, 0.0, 0.0, 1.0]
    return np.array(matmul3(Z, [float(v) for v in np.asarray(H, np.float64).reshape(9)])).reshape(3, 3)


def cropped_series(H_scaled, rows: int, cols: int, max_zoom: float, release: float, first_on: int = 0):
    """Hc and z of every call of a streaming run whose crop-off matrices are H_scaled[c] (call 0: identity) and whose crop
    was enabled before call `first_on` (earlier calls count as needing no zoom)."""
    R = crop_r(max_zoom, release)
    needs = [1.0 if c < first_on else need(H, rows, cols, max_zoom) for c, H in enumerate(H_scaled)]
    zs = schedule(needs, 0, len(needs), R, release, max_zoom)
    return [apply(z, H, rows, cols) for z, H in zip(zs, H_scaled)], zs
