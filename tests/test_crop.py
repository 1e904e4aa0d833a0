"""Auto-crop without a GPU: vstab_crop_zoom (the closed form the K16 kernel runs, csrc/homography.cuh) against the
restatement in tests/crop_ref.py and a brute-force coverage check, the causal zoom schedule across shard cuts, the fused
plan with the window widened by R, argument checks and the front ends' --crop flag."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import __graft_entry__ as entry
import crop_ref as cr
import vstab_b200 as vs

ROWS, COLS = 1080, 1920


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(vs.LIB_PATH):
        entry.build()
    return vs.load_library()


def _similarity(rng, scale=0.03, shift=40.0, persp=2e-6):
    s = 1.0 + rng.uniform(-scale, scale)
    a = rng.uniform(-0.03, 0.03)
    c0 = np.array([(COLS - 1) / 2, (ROWS - 1) / 2])
    H = np.eye(3)
    H[:2, :2] = s * np.array([[math.cos(a), -math.sin(a)], [math.sin(a), math.cos(a)]])
    H[:2, 2] = c0 - H[:2, :2] @ c0 + rng.uniform(-shift, shift, 2)
    H[2, :2] = rng.uniform(-persp, persp, 2)
    return H


def _rel(a, b):
    return abs(a - b) / abs(b)


def test_closed_form_equals_restatement(lib):
    rng = np.random.default_rng(7)
    for _ in range(500):
        H = _similarity(rng)
        for mz in (1.5, 4.0):
            got, want = vs.crop_zoom(H, ROWS, COLS, mz), cr.need(H, ROWS, COLS, mz)
            assert _rel(got, want) <= 1e-12, (H, got, want)
            assert 1.0 <= got <= mz


def test_identity_and_pure_shifts(lib):
    assert vs.crop_zoom(np.eye(3), ROWS, COLS, 4.0) == 1.0
    assert vs.crop_zoom(np.eye(3), 7, 5, 2.0) == 1.0
    half = (COLS - 1) / 2
    for dx in (0.25, 1.0, 17.5, -30.0, 200.0):
        H = np.eye(3)
        H[0, 2] = dx
        want = half / (half - abs(dx))
        assert _rel(vs.crop_zoom(H, ROWS, COLS, 4.0), want) <= 1e-12
        assert _rel(cr.need(H, ROWS, COLS, 4.0), want) <= 1e-12
        H = np.eye(3)
        H[1, 2] = dx                                   # vertical shifts: the same with rows
        want = ((ROWS - 1) / 2) / ((ROWS - 1) / 2 - abs(dx))
        assert _rel(vs.crop_zoom(H, ROWS, COLS, 4.0), want) <= 1e-12


def test_degenerate_matrices_need_max_zoom(lib):
    mz = 2.5
    flip_w = np.eye(3)
    flip_w[2] = [-1e-3, 0.0, 1.0]                      # w <= 0 at the right-hand corners
    far = np.eye(3)
    far[0, 2] = 5000.0                                 # the centre is outside H(S)
    nan = np.eye(3)
    nan[1, 1] = np.nan
    inf = np.eye(3)
    inf[0, 0] = np.inf
    flat = np.zeros((3, 3))
    flat[2, 2] = 1.0                                   # H(S) is one point
    for H in (flip_w, far, nan, inf, flat, -np.eye(3)):
        assert vs.crop_zoom(H, ROWS, COLS, mz) == mz
        assert cr.need(H, ROWS, COLS, mz) == mz
    big = np.eye(3)
    big[0, 2] = 900.0                                  # needs more than max_zoom: capped
    assert vs.crop_zoom(big, ROWS, COLS, 1.2) == 1.2


def _outside(Hc, pts):
    """how far (px) the source points Hc^-1(pts) of the output pixel centres pts fall outside S (0 when inside)"""
    src = np.linalg.inv(Hc) @ np.vstack([pts.T, np.ones(len(pts))])
    x, y = src[0] / src[2], src[1] / src[2]
    return max(float(np.max(-x)), float(np.max(x - (COLS - 1))), float(np.max(-y)), float(np.max(y - (ROWS - 1))), 0.0)


def test_brute_force_coverage():
    """The pixel centres of S, densely sampled (edges at every pixel, corners included): at need no warped sample reads
    outside S, at need * (1 - 1e-4) some does."""
    rng = np.random.default_rng(11)
    xs, ys = np.arange(COLS, dtype=float), np.arange(ROWS, dtype=float)
    edge = np.concatenate([np.stack([xs, np.zeros_like(xs)], 1), np.stack([xs, np.full_like(xs, ROWS - 1)], 1),
                           np.stack([np.zeros_like(ys), ys], 1), np.stack([np.full_like(ys, COLS - 1), ys], 1)])
    gx, gy = np.meshgrid(np.linspace(0, COLS - 1, 61), np.linspace(0, ROWS - 1, 35))
    pts = np.concatenate([edge, np.stack([gx.ravel(), gy.ravel()], 1)])
    checked = 0
    for _ in range(200):
        H = _similarity(rng)
        n = cr.need(H, ROWS, COLS, 4.0)
        if not 1.0 < n < 4.0:
            continue
        assert _outside(cr.apply(n, H, ROWS, COLS), pts) <= 1e-7
        assert _outside(cr.apply(n * (1 - 1e-4), H, ROWS, COLS), pts) > 1e-7
        checked += 1
    assert checked >= 150


def test_schedule_is_the_same_for_every_shard_cut():
    """z_c from the history of calls [c-R, c] only: shards [a, b) restated with the needs of [max(0, a-R), b) give the
    whole-clip schedule bit for bit."""
    rng = np.random.default_rng(3)
    for mz, rel in ((1.3, 0.002), (2.0, 0.05), (1.05, 0.01)):
        R = cr.crop_r(mz, rel)
        N = 600
        needs = [1.0] + list(np.minimum(mz, 1.0 + np.abs(rng.normal(0, (mz - 1) / 3, N - 1)) * (rng.random(N - 1) < 0.2)))
        whole = cr.schedule(needs, 0, N, R, rel, mz)
        assert whole[0] == 1.0 and max(whole) <= mz and min(whole) >= 1.0
        # falls by at most `release` per call, rises at once to what the call needs
        for c in range(1, N):
            assert whole[c] >= needs[c] and whole[c] >= whole[c - 1] - rel * (1 + 1e-12)
        cuts = sorted(set([0, N] + list(rng.integers(1, N, 7))))
        for a, b in zip(cuts[:-1], cuts[1:]):
            lo = max(0, a - R)
            part = cr.schedule(needs[lo:b], a, b - a, R, rel, mz, base=lo)
            assert part == whole[a:b], (mz, rel, a, b)


@pytest.mark.parametrize("N,world,P,F,B,R", [(1000, 2, 15, 15, 16, 100), (333, 8, 4, 3, 2, 50), (5000, 3, 60, 45, 128, 250),
                                             (97, 4, 1, 1, 3, 20)])
def test_fused_plan_with_window_widened_by_R(lib, N, world, P, F, B, R):
    """vstab_offline_run plans its fused pass with past P + R when the crop is on: every call is covered once, a fused call
    reads only its rank's own transforms, and ranks > 0 defer at most P+R-1 + F-1 calls to after the exchange."""
    seen = []
    for rank in range(world):
        pl, fp = vs.ShardPlan(), vs.FusedPlan()
        assert lib.vstab_offline_plan(N, world, rank, F, C.byref(pl)) == vs.OK
        assert lib.vstab_offline_fused_plan(N, world, rank, P + R, F, B, C.byref(fp)) == vs.OK
        assert pl.call_first <= fp.fused_first <= fp.fused_last <= pl.call_last
        seen += list(range(pl.call_first, pl.call_last))
        if fp.fused_last > fp.fused_first:
            assert pl.first == 0 or fp.fused_first - R - P - F + 1 >= pl.first
            assert fp.fused_last - 1 <= pl.last                      # its newest transform T[c-1] is the rank's own
        if rank > 0 and pl.call_last > pl.call_first:
            assert (fp.fused_first - pl.call_first) + (pl.call_last - fp.fused_last) <= (P + R - 1) + (F - 1)
        ref = vs.FusedPlan()
        assert lib.vstab_offline_fused_plan(N, world, rank, P, F, B, C.byref(ref)) == vs.OK
        assert ref.ring_chunks == fp.ring_chunks                     # the ring and (unless nothing is fused) the tail stay
        assert ref.fused_last == fp.fused_last or fp.fused_first == fp.fused_last
    assert seen == list(range(N))


def test_argument_checks(lib):
    assert lib.vstab_set_crop(None, 1.5, 0.01) == vs.ERR_INVALID_ARGUMENT
    assert lib.vstab_offline_set_crop(None, 1.5, 0.01) == vs.ERR_INVALID_ARGUMENT
    H = np.eye(3)
    p = H.ctypes.data_as(C.POINTER(C.c_double))
    for rows, cols, mz in ((1, 100, 2.0), (100, 1, 2.0), (0, 0, 2.0), (-5, 100, 2.0), (100, 100, 0.5), (100, 100, 4.5),
                           (100, 100, float("nan"))):
        assert lib.vstab_crop_zoom(p, rows, cols, mz) == -1.0
        with pytest.raises(ValueError):
            vs.crop_zoom(H, rows, cols, mz)
    assert lib.vstab_crop_zoom(None, 100, 100, 2.0) == -1.0
    assert lib.vstab_crop_zoom(p, 2, 2, 1.0) == 1.0


def _exe(name):
    exe = os.path.join(os.path.dirname(os.path.dirname(vs.LIB_PATH)), "bin", name)
    assert os.path.exists(exe), f"video-stabilization_b200/bin/{name} is built by make (__graft_entry__.build())"
    return exe


@pytest.mark.parametrize("name", ["vstab_file", "vstab_offline"])
def test_front_end_crop_flag(tmp_path, lib, name):
    """--crop MAX_ZOOM[,RELEASE]: malformed or out-of-range values are usage errors (exit status 1) before any device work;
    a valid one reaches the constructor's checks (workingHeight <= 90: exit 1 with its message)."""
    exe = _exe(name)
    clip = tmp_path / "c.bgr"
    clip.write_bytes(bytes(64 * 48 * 3))
    base = [exe, "--file", str(clip), "--out", str(tmp_path / "o.bgr"), "--width", "64", "--height", "48"]
    for bad in ("", "abc", "1.5,", ",0.01", "1.5,x", "1.5,0.01,2", "1.0", "0.5", "4.5", "nan", "1.5,0", "1.5,-0.01",
                "1.5,inf", "2,0.0001", "1.5x"):
        r = subprocess.run(base + ["--crop", bad], capture_output=True, text=True)
        assert r.returncode == 1 and "usage:" in r.stderr, (bad, r.returncode, r.stderr)
    r = subprocess.run(base + ["--crop"], capture_output=True, text=True)
    assert r.returncode == 1
    r = subprocess.run([exe, "--help"], capture_output=True, text=True)
    assert "--crop MAX_ZOOM[,RELEASE]" in r.stderr
    for good in ("1.2", "4,0.05", "1.5,0.002"):
        r = subprocess.run(base + ["--crop", good, "--working-height", "90"], capture_output=True, text=True)
        assert r.returncode == 1 and "workingHeight" in r.stderr, (good, r.stderr)
