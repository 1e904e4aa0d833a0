"""Auto-crop on the GPU (K16, vstab_set_crop / vstab_offline_set_crop): the matrices against the restatement in
tests/crop_ref.py fed with the oracle's crop-off H_stabilize_scaled, every output against cv2.warpPerspective of the presented
frame with the device's matrix, border-free outputs wherever the zoom is below its cap, offline == streaming through the
building blocks, run_host and vstab_offline_run, switches between calls, the trail, and crop off == never enabled."""
import numpy as np
import pytest

import crop_ref as cr
import vstab_b200 as vs
from conftest import render_clip
from oracle import stabilizer_ref as sr
from vstab_b200 import offline
from yuv_ref import NV12, bgr_to_yuv420, yuv420_to_bgr

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")
torch = pytest.importorskip("torch")

MZ, REL = 1.15, 0.004          # R = 38 calls: longer than every batch below
H_PX = 1e-9


def _corner_diff(Ha, Hb, W, H):
    c = np.array([[0, 0, 1], [W - 1, 0, 1], [0, H - 1, 1], [W - 1, H - 1, 1]], float).T
    a, b = Ha @ c, Hb @ c
    return float(np.abs(a[:2] / a[2] - b[:2] / b[2]).max())


def _warp(img, M, border):
    h, w = img.shape[:2]
    return cv2.warpPerspective(img, M, (w, h), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT,
                               borderValue=tuple(float(b) for b in border))


class _Restated:
    """z_c of a streaming run, call by call: needs from the oracle's crop-off H_scaled; (re)enabling the crop sets the
    history of the calls before it to 1."""

    def __init__(self, rows, cols):
        self.rows, self.cols, self.on, self.needs = rows, cols, None, {}

    def set(self, mz, rel, c):
        self.on = (mz, rel, cr.crop_r(mz, rel)) if mz > 1.0 else None
        self.needs = {j: 1.0 for j in range(max(c, 1))}          # call 0 (H = I) needs no zoom either

    def matrix(self, c, H):
        if self.on is None:
            return H, None
        mz, rel, R = self.on
        self.needs[c] = cr.need(H, self.rows, self.cols, mz)
        z = cr.zoom_at(self.needs, 0, c, R, rel, mz)
        return cr.apply(z, H, self.rows, self.cols), z


STREAM_CASES = {
    # name: (P, F, wh, W, H, n, script {call: ("mode", m) | ("crop", (mz, rel))})
    "global-F0": (5, 0, 135, 480, 270, 30, {0: ("crop", (MZ, REL)), 12: ("mode", sr.ACCUMULATED_FULL_LOCK), 20: ("mode", sr.GLOBAL_SMOOTHING)}),
    "global-F1": (5, 1, 135, 480, 270, 30, {0: ("crop", (MZ, REL)), 14: ("mode", sr.ACCUMULATED_FULL_LOCK)}),
    "global-F9": (5, 9, 135, 480, 270, 34, {3: ("crop", (MZ, REL)), 16: ("mode", sr.ACCUMULATED_FULL_LOCK)}),
    "lock-F1": (5, 1, 135, 480, 270, 40, {0: ("crop", (MZ, REL)), 6: ("mode", sr.ACCUMULATED_FULL_LOCK)}),
    "lock-F9": (5, 9, 135, 480, 270, 40, {0: ("crop", (MZ, 0.02)), 10: ("mode", sr.ACCUMULATED_FULL_LOCK)}),
    "orb-F3": (5, 3, 360, 640, 360, 22, {0: ("crop", (MZ, REL)), 6: ("mode", sr.ORB_FULL_LOCK)}),
}


@pytest.mark.parametrize("case", sorted(STREAM_CASES))
def test_streaming_crop_against_oracle(texture_small, case):
    P, F, wh, W, H, n, script = STREAM_CASES[case]
    frames = render_clip(texture_small, W, H, n)
    ref = sr.StabilizerRef(P, F, wh)
    st = vs.Stabilizer(P, F, wh)
    rs = _Restated(H, W)
    needs, zs = [], []
    for i, f in enumerate(frames):
        if i in script:
            what, v = script[i]
            if what == "mode":
                ref.set_stabilization_mode(v); st.set_stabilization_mode(v)
            else:
                st.set_crop(*v); rs.set(*v, i)
        want = ref.stabilize_frame(f)
        got = st.stabilize_frame(f)
        if i == 0:
            assert np.array_equal(got, f)                          # call 0: the copy of its input, H = I, z = 1
            continue
        H_ref = ref.taps.H_scaled
        H_want, z = rs.matrix(i, H_ref)
        got_H = st.tap(vs.TAP_H_SCALED)
        assert _corner_diff(got_H, H_want, W, H) <= H_PX, (i, z)
        assert _corner_diff(st.tap(vs.TAP_H_STABILIZE), ref.taps.H_stabilize, W, H) <= H_PX   # uncropped working H
        pres = frames[st.presentation_index()]
        border = st.tap(vs.TAP_BORDER)
        assert np.array_equal(got, _warp(pres, got_H, border)), i
        avg = tuple(0.5 * v for v in cv2.mean(pres))
        assert int(np.abs(got.astype(int) - _warp(pres, H_want, avg)).max()) <= 1, i
        if z is not None:
            needs.append(rs.needs[i]); zs.append(z)
            if z < rs.on[0]:                                       # border-free below the cap
                black, white = _warp(pres, got_H, (0, 0, 0)), _warp(pres, got_H, (255, 255, 255))
                assert np.array_equal(black, white) and np.array_equal(got, black), (i, z)
    st.close()
    assert zs and min(zs) >= 1.0
    if case.startswith("lock"):
        assert max(needs) > 1.1 and max(zs) == MZ                  # drift large enough to reach the cap
    else:
        assert max(zs) > 1.01


def test_switches_trail_and_restatement(texture_small):
    """Crop on / off / re-enabled with other parameters between calls, mixed with mode and trail switches: each switch drops
    the output prepared one call ahead; every matrix matches the restatement and every output is the warp (or, with the
    trail, copyFeathered over the previous output) of the presented frame by the device's matrix."""
    W, H, n = 480, 270, 44
    frames = render_clip(texture_small, W, H, n)
    ref = sr.StabilizerRef(5, 3, 135)
    st = vs.Stabilizer(5, 3, 135)
    rs = _Restated(H, W)
    script = {2: ("crop", (MZ, REL)), 8: ("mode", sr.ACCUMULATED_FULL_LOCK), 11: ("trail", True), 15: ("crop", (1.0, 0.0)),
              17: ("trail", False), 19: ("crop", (1.3, 0.01)), 21: ("mode", sr.GLOBAL_SMOOTHING), 24: ("trail", True),
              27: ("trail", False), 29: ("crop", (1.0, 0.0)), 30: ("crop", (1.08, 0.002)), 33: ("mode", sr.ACCUMULATED_FULL_LOCK),
              38: ("crop", (1.08, 0.002))}
    trail, bg = False, np.zeros((H, W, 3), np.uint8)               # the trail background: zeros, then each trail output
    for i, f in enumerate(frames):
        if i in script:
            what, v = script[i]
            if what == "mode":
                ref.set_stabilization_mode(v); st.set_stabilization_mode(v)
            elif what == "trail":
                trail = v; st.set_trail(v)
            else:
                st.set_crop(*v); rs.set(*v, i)
        ref.stabilize_frame(f)
        got = st.stabilize_frame(f)
        if i:
            H_want, z = rs.matrix(i, ref.taps.H_scaled)
            got_H = st.tap(vs.TAP_H_SCALED)
            assert _corner_diff(got_H, H_want, W, H) <= H_PX, i
            pres = frames[st.presentation_index()]
            if trail:
                assert np.array_equal(got, vs.k_copy_feathered(pres, bg, got_H)), i
            else:
                assert np.array_equal(got, _warp(pres, got_H, st.tap(vs.TAP_BORDER))), i
        if trail:
            bg = got.copy()
    st.close()


def test_crop_off_equals_never_enabled(texture_small):
    """set_crop(...) then set_crop(1.0, 0): the same bytes and the same launches per call as an instance that never had it."""
    frames = render_clip(texture_small, 480, 270, 20)
    runs = []
    for enable in (True, False):
        st = vs.Stabilizer(5, 3, 135)
        if enable:
            st.set_crop(1.3, 0.01)
            st.set_crop(1.0, 0.0)
        outs, deltas = [], []
        lib = vs.load_library()
        for i, f in enumerate(frames):
            if i == 9:
                st.set_stabilization_mode(vs.ACCUMULATED_FULL_LOCK)
            l0 = lib.vstab_launch_count()
            outs.append(st.stabilize_frame(f))
            deltas.append(lib.vstab_launch_count() - l0)
        st.close()
        runs.append((outs, deltas))
    assert runs[0][1] == runs[1][1]
    for a, b in zip(runs[0][0], runs[1][0]):
        assert np.array_equal(a, b)


def test_argument_errors():
    st = vs.Stabilizer(3, 2, 135)
    off = offline.OfflineStabilizer(3, 2, 135, 270, 480, 4)
    for mz, rel in ((0.5, 0.01), (4.5, 0.01), (1.5, 0.0), (1.5, -0.01), (float("nan"), 0.01), (1.5, float("nan")),
                    (1.5, float("inf")), (2.0, 1e-4), (-1.0, 0.01)):
        with pytest.raises(ValueError):
            st.set_crop(mz, rel)
        with pytest.raises(ValueError):
            off.set_crop(mz, rel)
    st.set_crop(4.0, 0.001)                                       # R = 3000: accepted
    off.set_crop(4.0, 0.001)
    st.close()
    off.close()


# ---- offline == streaming ----------------------------------------------------------------------------------------------
def _dev_clip(tex_np, W, H, n):
    from oracle import synth
    tex = torch.from_numpy(tex_np).cuda()
    path = synth.camera_path(n)
    out = torch.empty((n, H, W, 3), dtype=torch.uint8, device="cuda")
    offline.render_frames(tex, path, H, W, synth.focal_for_width(W), out)
    return out, path, tex


def _streaming(frames_np, P, F, wh, lock_at, crop):
    st = vs.Stabilizer(P, F, wh)
    st.set_crop(*crop)
    outs, Hs = [], []
    for i, f in enumerate(frames_np):
        if lock_at is not None and i == lock_at:
            st.set_stabilization_mode(vs.ACCUMULATED_FULL_LOCK)
        outs.append(st.stabilize_frame(f))
        Hs.append(st.tap(vs.TAP_H_SCALED) if i else np.eye(3))
    st.close()
    return outs, Hs


W0, H0, WH0, P0, F0, N0 = 480, 270, 135, 6, 4, 60


@pytest.fixture(scope="module")
def clip(texture_small):
    frames, path, tex = _dev_clip(texture_small, W0, H0, N0)
    f_np = np.ascontiguousarray(frames.cpu().numpy())
    want = {lock: _streaming(f_np, P0, F0, WH0, lock, (MZ, REL)) for lock in (None, 9)}
    return frames, f_np, path, tex, want


@pytest.mark.parametrize("lock_at", [None, 9])
@pytest.mark.parametrize("shards", [[(0, N0)], [(0, 30), (30, N0)], [(0, 7), (7, 41), (41, N0)]])
def test_building_blocks_equal_streaming(clip, lock_at, shards):
    """estimate / prepare / render per shard, in batches of 7 calls (< R = 38): every render recomputes its halo calls."""
    frames, f_np, _, _, want = clip
    want_out, want_H = want[lock_at]
    mode = vs.GLOBAL_SMOOTHING if lock_at is None else vs.ACCUMULATED_FULL_LOCK
    T_parts, sums_parts, runners = [], [], []
    for (first, last) in shards:
        off = offline.OfflineStabilizer(P0, F0, WH0, H0, W0, 7)
        off.set_crop(MZ, REL)
        T = torch.zeros((last - first, 9), dtype=torch.float64, device="cuda")
        sums = torch.zeros((last - first, 3), dtype=torch.int64, device="cuda")
        off.estimate(frames[first:last], first, frames[first - 1] if first else None, T, sums)
        off.synchronize()
        T_parts.append(T); sums_parts.append(sums); runners.append(off)
    T_all = torch.cat(T_parts, 0)
    seen = []
    for (first, last), sums, off in zip(shards, sums_parts, runners):
        c0, c1 = offline.calls_of_shard(first, last, N0, F0)
        out = torch.empty((max(c1 - c0, 1), H0, W0, 3), dtype=torch.uint8, device="cuda")
        off.prepare(T_all, mode, lock_at or 0)
        done = 0
        while done < c1 - c0:
            m = min(7, c1 - c0 - done)
            off.render(frames[first:last], first, c0 + done, m, T_all, mode, lock_at or 0, sums, out[done:])
            hs = off.read_h(m)
            o = out[done:done + m].cpu().numpy()
            for j in range(m):
                c = c0 + done + j
                assert np.array_equal(o[j], want_out[c]), c
                if c:
                    assert np.array_equal(hs[j], want_H[c]), c
                seen.append(c)
            done += m
        off.close()
    assert seen == list(range(N0))


@pytest.mark.parametrize("yuv", [False, True])
def test_run_host_equals_streaming(clip, yuv):
    frames, f_np, _, _, want = clip
    off = offline.OfflineStabilizer(P0, F0, WH0, H0, W0, 7)
    off.set_crop(MZ, REL)
    if yuv:
        off.set_yuv(vs.PIX_NV12, vs.PIX_NV12)
        src = np.ascontiguousarray(np.stack([bgr_to_yuv420(f, NV12) for f in f_np]))
        exp = [bgr_to_yuv420(o, NV12) for o in
               _streaming(np.stack([yuv420_to_bgr(s, NV12) for s in src]), P0, F0, WH0, None, (MZ, REL))[0]]
    else:
        src, exp = f_np, want[None][0]
    out = np.zeros_like(src)
    off.run_host(src.ctypes.data, src.strides[0], src.strides[1], N0, vs.GLOBAL_SMOOTHING, 0, out.ctypes.data,
                 out.strides[0], out.strides[1])
    off.close()
    for c in range(N0):
        assert np.array_equal(out[c], exp[c]), c


@pytest.mark.parametrize("B", [2, 3, 16])
@pytest.mark.parametrize("source", ["host", "device", "sim"])
@pytest.mark.parametrize("lock_at", [None, 9])
def test_offline_run_equals_streaming(clip, B, source, lock_at):
    """vstab_offline_run as a world of one: GLOBAL_SMOOTHING from host / simulator frames is the fused pass, the device
    source and the lock mode the two-pass job.  R = 38 is larger than every batch."""
    frames, f_np, path, tex, want = clip
    from oracle import synth
    mode = vs.GLOBAL_SMOOTHING if lock_at is None else vs.ACCUMULATED_FULL_LOCK
    off = offline.OfflineStabilizer(P0, F0, WH0, H0, W0, B)
    off.set_crop(MZ, REL)
    off.comm_init(0, 1)
    kw = {"host": dict(host_frames=f_np), "device": dict(device_frames=frames),
          "sim": dict(texture=tex, poses=path, focal=synth.focal_for_width(W0))}[source]
    dout = torch.empty((N0, H0, W0, 3), dtype=torch.uint8, device="cuda") if source == "device" else None
    r = off.run(N0, mode, lock_at or 0, device_out=dout, **kw)
    off.close()
    assert list(r["checksums"]) == [vs.frame_checksum(o) for o in want[lock_at][0]]
    if dout is not None:
        got = dout.cpu().numpy()
        for c in range(N0):
            assert np.array_equal(got[c], want[lock_at][0][c]), c
