"""Float64 restatement of K6 (csrc/smooth.cu): window average, accumulated lock, mode selection, translation rescale
and border colour, in plain Python floats, one IEEE operation at a time and in smooth.cu's order.

smooth.cu is compiled with -fmad=false and spells out its operation order, so the device results equal these bit for
bit; only device sin / cos / atan2 (the partial-lock rotation) may differ from libm by an ulp.  No test functions here:
tests/test_trajectory.py checks this module against the oracle and mpmath, tests/test_gpu_trajectory.py checks the
kernels against it.

Index algebra (SURVEY Appendix C): call c presents frame p = max(0, c - F) from the window [lo, c],
lo = max(0, c - W + 1), W = P + 1 + F; T[k] maps frame k - 1 to frame k.
"""
import math

import numpy as np

from oracle.stabilizer_ref import decompose_homography

ACCUMULATED_FULL_LOCK, TRANSLATION_LOCK, ROTATION_LOCK, GLOBAL_SMOOTHING = 0, 3, 4, 5

I3 = (1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0)


def matmul3(A, B):
    """C = A @ B, each entry s = a*b; s = s + a*b; s = s + a*b (homography.cuh matmul3)."""
    a0, a1, a2, a3, a4, a5, a6, a7, a8 = A
    b0, b1, b2, b3, b4, b5, b6, b7, b8 = B
    return [a0 * b0 + a1 * b3 + a2 * b6, a0 * b1 + a1 * b4 + a2 * b7, a0 * b2 + a1 * b5 + a2 * b8,
            a3 * b0 + a4 * b3 + a5 * b6, a3 * b1 + a4 * b4 + a5 * b7, a3 * b2 + a4 * b5 + a5 * b8,
            a6 * b0 + a7 * b3 + a8 * b6, a6 * b1 + a7 * b4 + a8 * b7, a6 * b2 + a7 * b5 + a8 * b8]


def invert3(a):
    """(ok, inverse): cofactors times 1/det; (False, zeros) when det == 0 (homography.cuh invert3, cv::invert)."""
    a0, a1, a2, a3, a4, a5, a6, a7, a8 = a
    d = a0 * (a4 * a8 - a5 * a7) - a1 * (a3 * a8 - a5 * a6) + a2 * (a3 * a7 - a4 * a6)
    if d == 0.0:
        return False, [0.0] * 9
    d = 1.0 / d
    return True, [(a4 * a8 - a5 * a7) * d, (a2 * a7 - a1 * a8) * d, (a1 * a5 - a2 * a4) * d,
                  (a5 * a6 - a3 * a8) * d, (a0 * a8 - a2 * a6) * d, (a2 * a3 - a0 * a5) * d,
                  (a3 * a7 - a4 * a6) * d, (a1 * a6 - a0 * a7) * d, (a0 * a4 - a1 * a3) * d]


def finite9(H):
    return all(math.isfinite(v) for v in H)


def window(c, P, F):
    """(lo, p) of call c"""
    W = P + 1 + F
    return max(0, c - W + 1), max(0, c - F)


def window_average(T, c, P, F):
    """The GLOBAL_SMOOTHING matrix of call c: past chain acc = inv(T[k]) @ acc for k = p .. lo+1 and future chain
    acc = acc @ T[k] for k = p+1 .. c-1, each summed term by term, then (past_sum + future_sum) / count.
    Identity when count == 0 or the average is not finite.  T[k]: 9 floats."""
    lo, p = window(c, P, F)
    past = [0.0] * 9
    n = 0
    acc = I3
    for k in range(p, lo, -1):
        acc = matmul3(invert3(T[k])[1], acc)
        past = [s + x for s, x in zip(past, acc)]
        n += 1
    fut = [0.0] * 9
    acc = I3
    for k in range(p + 1, c):
        acc = matmul3(acc, T[k])
        fut = [s + x for s, x in zip(fut, acc)]
        n += 1
    if n == 0:
        return list(I3)
    avg = [(s + f) / n for s, f in zip(past, fut)]
    return avg if finite9(avg) else list(I3)


def accumulated(T, anchor, n_total):
    """acc[anchor] = I, acc[k] = T[k] @ acc[k-1] for k < n_total (acc_seq_kernel, acc_update_kernel); None before."""
    acc = [None] * n_total
    if anchor < n_total:
        acc[anchor] = list(I3)
        for k in range(anchor + 1, n_total):
            acc[k] = matmul3(T[k], acc[k - 1])
    return acc


def lock_matrix(acc_p):
    """(H, theta): inverse of the accumulated product, identity (theta 0) when it does not decompose."""
    H = invert3(acc_p)[1]
    hp = decompose_homography(np.array(H).reshape(3, 3))
    if hp is None:
        return list(I3), 0.0
    return H, hp.theta


def partial_lock(Hl, theta, mode, cx, cy):
    """TRANSLATION_LOCK: R @ Hl, ROTATION_LOCK: inv(R), R = cv::getRotationMatrix2D((cx, cy), theta in degrees, 1)."""
    k_deg_to_rad = 3.1415926535897932384626433832795 / 180.0
    ang = (theta * 180.0 / 3.14159265358979323846) * k_deg_to_rad
    al, be = math.cos(ang), math.sin(ang)
    R = [al, be, (1.0 - al) * cx - be * cy, -be, al, be * cx + (1.0 - al) * cy, 0.0, 0.0, 1.0]
    return matmul3(R, Hl) if mode == TRANSLATION_LOCK else invert3(R)[1]


def border(sums, npix):
    """saturate_cast<uchar>(0.5 * mean) per channel: round half to even, clamped to 0..255."""
    return [min(255, max(0, round(0.5 * (float(s) / npix)))) for s in sums]


def call_params(T, c, P, F, mode, *, lock_call=0, acc=None, scale=1.0, sums=None, npix=1.0, partial_fix=False,
                cx=0.0, cy=0.0):
    """What smooth_kernel writes for call c: dict(p, Hw (working resolution), Hs (translation rescaled), border).
    `acc[p]`: accumulated product of the presented frame (ACCUMULATED_FULL_LOCK / partial lock); `sums`: channel
    sums of the presented frame."""
    assert mode in (ACCUMULATED_FULL_LOCK, TRANSLATION_LOCK, ROTATION_LOCK, GLOBAL_SMOOTHING)
    _, p = window(c, P, F)
    if mode == ACCUMULATED_FULL_LOCK and c < lock_call:
        mode = GLOBAL_SMOOTHING                            # the window average until the lock call
    partial = partial_fix and mode in (TRANSLATION_LOCK, ROTATION_LOCK)
    if mode == GLOBAL_SMOOTHING:
        H = window_average(T, c, P, F)
    elif mode == ACCUMULATED_FULL_LOCK or partial:
        H, theta = lock_matrix(acc[p])
        if partial:
            H = partial_lock(H, theta, mode, cx, cy)
    else:
        H = list(I3)                                       # T / R lock as the reference ships it: identity
    Hw = list(H)
    if abs(scale - 1.0) > 1e-6:
        H[2] /= scale
        H[5] /= scale
    return dict(p=p, Hw=Hw, Hs=H, border=border(sums, npix) if sums is not None else None)


def corner_diff(A, B, w, h):
    """largest distance between the images of the frame corners under A and B, px"""
    corners = np.array([[0, 0, 1], [w, 0, 1], [0, h, 1], [w, h, 1]], float).T
    a = np.asarray(A, float).reshape(3, 3) @ corners
    b = np.asarray(B, float).reshape(3, 3) @ corners
    return float(np.abs(a[:2] / a[2] - b[:2] / b[2]).max())


# ---- seeded transform families (T[0] is never read: the identity) ---------------------------------------------------
def _similarity(th, tx, ty):
    c, s = math.cos(th), math.sin(th)
    return [c, -s, float(tx), s, c, float(ty), 0.0, 0.0, 1.0]


def transforms(kind, n, seed):
    """n transforms T[0..n) of one family, as lists of 9 floats.
    walk:   similarity random walk (0.01 rad, 3 px per step), what the fit produces on a handheld clip
    large:  T[k] = J[k] @ inv(J[k-1]) for independent poses J of up to 1 rad and 1e3 px (large, bounded motion)
    affine: walk with shear / anisotropic scale of 1e-3 and projective terms of 1e-6"""
    rng = np.random.default_rng(seed)
    T = [list(I3)]
    if kind == "walk":
        for _ in range(1, n):
            th, tx, ty = float(rng.normal(0, 0.01)), *rng.normal(0, 3, 2)
            T.append(_similarity(th, tx, ty))
    elif kind == "large":
        J = [_similarity(float(rng.uniform(-1, 1)), *rng.uniform(-1e3, 1e3, 2)) for _ in range(n)]
        for k in range(1, n):
            T.append(matmul3(J[k], invert3(J[k - 1])[1]))
    elif kind == "affine":
        for _ in range(1, n):
            th, tx, ty = float(rng.normal(0, 0.01)), *rng.normal(0, 3, 2)
            m = _similarity(th, tx, ty)
            e = rng.normal(0, 1e-3, 4)
            m[0] += float(e[0]); m[1] += float(e[1]); m[3] += float(e[2]); m[4] += float(e[3])
            m[6], m[7] = (float(v) for v in rng.normal(0, 1e-6, 2))
            T.append(m)
    else:
        raise ValueError(kind)
    return T
