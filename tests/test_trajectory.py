"""The K6 restatement (tests/trajectory_ref.py) against the oracle's own order (StabilizerRef._global_smoothing with
cv2.invert and numpy products) and against mpmath at 40-50 digits: the float64 chains the reference and the kernels
run do not drift over long windows and long clips.  CPU only."""
from collections import deque

import cv2
import numpy as np
import pytest

import trajectory_ref as tr
from oracle import stabilizer_ref as sr

mpmath = pytest.importorskip("mpmath")

W_PX, H_PX = 320, 180
# corner error bounds, px: the "large" family moves by up to 1e3 px a frame, so its last bits weigh 100x more
TOL = {"walk": 1e-11, "affine": 1e-11, "large": 1e-10}


def _oracle_average(T, c, P, F):
    lo, p = tr.window(c, P, F)
    o = sr.StabilizerRef(P, F, H_PX)
    o.transforms = deque((np.array(T[k]).reshape(3, 3), k - 1, k) for k in range(lo + 1, c + 1))
    return o._global_smoothing(p - lo)


def _calls(n, P, F, stride):
    """every call of the warm-up and around the first full window, then every `stride`-th call"""
    W = P + 1 + F
    edge = set(range(0, min(n, F + 3))) | set(range(max(0, W - 3), min(n, W + 3)))
    return sorted(edge | set(range(0, n, stride)) | {n - 1})


@pytest.mark.parametrize("P,F,n,stride,kind", [(5, 3, 60, 1, "walk"), (200, 100, 700, 7, "walk"), (300, 300, 700, 23, "walk"),
                                                 (300, 0, 500, 17, "affine"), (0, 300, 500, 17, "large"),
                                                 (128, 129, 400, 11, "large")])
def test_window_average_equals_oracle_order(P, F, n, stride, kind):
    """Same sums in the reference's order: the two differ only in the last bits of the products (cv2.invert / numpy
    matmul against the closed forms), <= 1e-11 px at the corners of a 320x180 frame for small motion."""
    T = tr.transforms(kind, n, seed=P * 1000 + F)
    worst = 0.0
    for c in _calls(n, P, F, stride):
        worst = max(worst, tr.corner_diff(tr.window_average(T, c, P, F), _oracle_average(T, c, P, F), W_PX, H_PX))
    assert worst <= TOL[kind], worst


def _mp(t):
    return mpmath.matrix([[mpmath.mpf(t[3 * i + j]) for j in range(3)] for i in range(3)])


def _mp_to_np(m):
    return np.array([[float(m[i, j]) for j in range(3)] for i in range(3)])


@pytest.mark.parametrize("P,F,kind", [(200, 100, "walk"), (300, 300, "affine"), (150, 120, "large")])
def test_window_average_equals_mpmath(P, F, kind):
    """The float64 window average against the exact average at 40 digits: <= 1e-11 px (measured ~1e-12)."""
    n = P + F + 40
    T = tr.transforms(kind, n, seed=7 + P)
    worst = 0.0
    with mpmath.workdps(40):
        for c in (F + 1, P + F // 2, P + F, n - 1):
            lo, p = tr.window(c, P, F)
            s, acc = mpmath.zeros(3, 3), mpmath.eye(3)
            for k in range(p, lo, -1):
                acc = _mp(T[k]) ** -1 * acc
                s += acc
            acc = mpmath.eye(3)
            for k in range(p + 1, c):
                acc = acc * _mp(T[k])
                s += acc
            want = _mp_to_np(s / ((p - lo) + max(0, c - 1 - p)))
            worst = max(worst, tr.corner_diff(tr.window_average(T, c, P, F), want, W_PX, H_PX))
    assert worst <= TOL[kind], worst


def test_accumulated_lock_3000_frames_equals_mpmath():
    """inv(acc[k]) of the sequential float64 prefix over a 3000-frame clip against the exact product at 50 digits:
    <= 1e-10 px (measured ~1e-12), so the reference's own lock chain does not drift."""
    n, anchor = 3000, 0
    T = tr.transforms("walk", n, seed=2)
    acc = tr.accumulated(T, anchor, n)
    worst = 0.0
    with mpmath.workdps(50):
        m = mpmath.eye(3)
        for k in range(anchor + 1, n):
            m = _mp(T[k]) * m
            if k % 250 == 0 or k == n - 1:
                H, _ = tr.lock_matrix(acc[k])
                worst = max(worst, tr.corner_diff(H, _mp_to_np(m ** -1), W_PX, H_PX))
    assert worst <= 1e-10, worst


def test_accumulated_lock_equals_oracle_order():
    """The restated lock against StabilizerRef._full_lock call by call (numpy products, cv2.invert)."""
    P, F, lock_call, n = 6, 4, 9, 300
    T = tr.transforms("affine", n, seed=3)
    o = sr.StabilizerRef(P, F, H_PX)
    o.set_stabilization_mode(sr.ACCUMULATED_FULL_LOCK)
    acc = tr.accumulated(T, lock_call - F, n)
    worst = 0.0
    for c in range(lock_call, n):
        lo, p = tr.window(c, P, F)
        o.frames = deque((None, k) for k in range(lo, c + 1))
        o.transforms = deque((np.array(T[k]).reshape(3, 3), k - 1, k) for k in range(lo + 1, c + 1))
        want = o._full_lock(p - lo)
        got = tr.call_params(T, c, P, F, tr.ACCUMULATED_FULL_LOCK, lock_call=lock_call, acc=acc)["Hs"]
        worst = max(worst, tr.corner_diff(got, want, W_PX, H_PX))
    assert worst <= 1e-11, worst


def test_fallbacks():
    """count == 0, a non-finite average and a lock that does not decompose give the identity; a window without the
    non-finite transform is unaffected."""
    T = tr.transforms("walk", 40, seed=5)
    assert tr.window_average(T, 0, 5, 3) == list(tr.I3)          # call 0: no terms
    assert tr.window_average(T, 1, 5, 3) == list(tr.I3)          # call 1, F >= 1: the newest transform is excluded
    assert tr.window_average(T, 1, 5, 0) != list(tr.I3)          # F == 0: one past term
    T[20] = [float("nan")] + T[20][1:]
    for c in range(21, 28):                                       # T[lo+1 .. c-1] holds T[20]
        assert tr.window_average(T, c, 5, 3) == list(tr.I3), c
    assert tr.window_average(T, 28, 5, 3) != list(tr.I3)          # lo = 20: T[20] has left the window
    T[30] = [1.0, 0.0, float("inf"), 0.0, 1.0, 0.0, 0.0, 0.0, 1.0]
    assert tr.window_average(T, 33, 5, 3) == list(tr.I3)
    acc = tr.accumulated(T, 10, 40)
    assert tr.call_params(T, 23, 5, 3, tr.ACCUMULATED_FULL_LOCK, lock_call=13, acc=acc)["Hs"] == list(tr.I3)   # p = 20
    assert tr.call_params(T, 22, 5, 3, tr.ACCUMULATED_FULL_LOCK, lock_call=13, acc=acc)["Hs"] != list(tr.I3)   # p = 19
    assert tr.lock_matrix([0.0] * 9) == (list(tr.I3), 0.0)       # singular: invert3 gives zeros, h33 == 0


def test_border_rounding_and_saturation():
    """0.5 * mean rounds half to even (saturate_cast<uchar> = cvRound) and saturates at 255."""
    npix = 96 * 128
    assert tr.border([3 * npix, 5 * npix, 1 * npix], npix) == [2, 2, 0]       # 1.5 -> 2, 2.5 -> 2, 0.5 -> 0
    assert tr.border([509 * npix, 510 * npix, 511 * npix], npix) == [254, 255, 255]
    assert tr.border([2 ** 40, 0, 3 * npix + 1], npix) == [255, 0, 2]
    assert tr.border([int(2.7 * npix)], npix) == [1]                             # 1.35 -> 1
    assert tr.border([int(3.4 * npix)], npix) == [2]                             # 1.7 -> 2


def test_partial_lock_matches_oracle():
    """The restated partial-lock R (smooth.cu:113-121) against StabilizerRef with partial_lock_fix (cv2.getRotationMatrix2D,
    cv2.invert)."""
    P, F, n = 6, 4, 120
    T = tr.transforms("walk", n, seed=11)
    cx, cy = float(np.float32(W_PX / 2.0)), float(np.float32(H_PX / 2.0))
    for mode in (tr.TRANSLATION_LOCK, tr.ROTATION_LOCK):
        acc = tr.accumulated(T, 9 - F, n)
        worst = 0.0
        for c in (9, 10, 50, n - 1):
            _, p = tr.window(c, P, F)
            Hl, _ = tr.lock_matrix(acc[p])
            hp = sr.decompose_homography(np.array(Hl).reshape(3, 3))
            R = np.eye(3)
            R[:2] = cv2.getRotationMatrix2D((cx, cy), hp.theta * 180.0 / np.pi, 1.0)
            want = R @ np.array(Hl).reshape(3, 3) if mode == tr.TRANSLATION_LOCK else np.linalg.inv(R)
            got = tr.call_params(T, c, P, F, mode, acc=acc, partial_fix=True, cx=cx, cy=cy)["Hs"]
            worst = max(worst, tr.corner_diff(got, want, W_PX, H_PX))
        assert worst <= 1e-9, (mode, worst)
