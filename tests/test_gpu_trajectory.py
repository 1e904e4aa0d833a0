"""K6 (csrc/smooth.cu: smooth_kernel, acc_seq_kernel, acc_update_kernel) against its float64 restatement
(tests/trajectory_ref.py), bit for bit, where the rest of the suite does not reach: windows longer than the 256 terms
smooth_kernel stages in shared memory, accumulated-lock clips over many 256-transform scan chunks with the anchor on and
off a chunk start, deep rings of the fused offline pass, non-finite transforms, and border colours on .5 ties and above
255.  The offline cases feed synthetic transforms and channel sums straight to vstab_offline_prepare / _render, so the
window and the lock are checked on inputs the fit would rarely produce; the output bytes are checked against
cv2.warpPerspective of the frame the restatement says is presented, with its border colour."""
import cv2
import numpy as np
import pytest

import trajectory_ref as tr
import vstab_b200 as vs
from conftest import render_clip
from vstab_b200 import offline

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

SMALL = (96, 128, 96)          # rows, cols, working height: scale 1
HALF = (192, 256, 96)          # scale 0.5: translations of Hs are rescaled


def _bits(H):
    return np.ascontiguousarray(np.asarray(H, np.float64).reshape(9)).view(np.uint64)


def _assert_bits(got, want, what):
    if not np.array_equal(_bits(got), _bits(want)):
        raise AssertionError(f"{what}: device H differs from the restatement "
                             f"(corner diff {tr.corner_diff(got, want, 320, 180):.3e} px)\n{np.reshape(got, (3, 3))}\n"
                             f"{np.reshape(want, (3, 3))}")


def _noise_frames(n, rows, cols, seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return torch.randint(0, 256, (n, rows, cols, 3), dtype=torch.uint8, device="cuda", generator=g)


def _sums(n, npix, seed):
    """channel sums: random means, exact odd means (0.5 * mean on a .5 tie), and sums far above 255 per pixel"""
    rng = np.random.default_rng(seed)
    s = rng.integers(0, 256 * npix, (n, 3), dtype=np.int64)
    ties = rng.random((n, 3)) < 0.3
    s[ties] = (2 * rng.integers(0, 255, int(ties.sum())) + 1) * npix
    sat = rng.random((n, 3)) < 0.15
    s[sat] = rng.integers(510 * npix, 2 ** 40, int(sat.sum()))
    return s


def _with_nonfinite(T, at, kind):
    T = [list(t) for t in T]
    T[at][2 if kind == "inf" else 0] = float(kind)
    return T


def _offline_check(frames, T, sums, shards, P, F, wh, mode, lock_call=0, batch=64):
    """Renders every call of the clip shard by shard (ranks emulated one after the other on this GPU, the gather is
    the shared T), and checks each call's Hs (read_h) and output bytes against the restatement."""
    n, rows, cols = frames.shape[0], frames.shape[1], frames.shape[2]
    scale, npix = wh / rows, float(rows * cols)
    T_all = torch.tensor(np.asarray(T, np.float64).reshape(n, 9), device="cuda")
    sums_all = torch.tensor(sums, device="cuda")
    acc = tr.accumulated(T, lock_call - F, n) if mode == tr.ACCUMULATED_FULL_LOCK else None
    frames_np = frames.cpu().numpy()
    seen = []
    for first, last in shards:
        off = offline.OfflineStabilizer(P, F, wh, rows, cols, batch)
        c0, c1 = offline.calls_of_shard(first, last, n, F)
        off.prepare(T_all, mode, lock_call)
        loc, loc_sums = frames[first:last], sums_all[first:last]
        out = torch.empty((batch, rows, cols, 3), dtype=torch.uint8, device="cuda")
        for b0 in range(c0, c1, batch):
            m = min(batch, c1 - b0)
            off.render(loc, first, b0, m, T_all, mode, lock_call, loc_sums, out)
            hs = off.read_h(m)
            got = out[:m].cpu().numpy()
            for j in range(m):
                c = b0 + j
                want = tr.call_params(T, c, P, F, mode, lock_call=lock_call, acc=acc, scale=scale, sums=sums[max(0, c - F)],
                                      npix=npix)
                _assert_bits(hs[j], want["Hs"], f"call {c}")
                ref = cv2.warpPerspective(frames_np[want["p"]], np.reshape(want["Hs"], (3, 3)), (cols, rows), flags=cv2.INTER_LINEAR,
                                          borderMode=cv2.BORDER_CONSTANT, borderValue=tuple(float(v) for v in want["border"]))
                assert np.array_equal(got[j], ref), f"call {c}: output bytes (presented frame {want['p']})"
                seen.append(c)
        off.close()
    assert sorted(seen) == list(range(n))


@pytest.mark.parametrize("P,F,geom", [(128, 129, SMALL), (129, 129, HALF), (300, 200, SMALL), (300, 0, HALF),
                                      (0, 300, SMALL)])
def test_window_average_across_the_staging_limit(P, F, geom):
    """P + F - 1 = 256 terms (the largest window smooth_kernel stages in shared memory), 257 (the first one read from
    global memory), and 300/200, 300/0 and 0/300, whose warm-up calls cross 256 terms on the way."""
    rows, cols, wh = geom
    n = P + F + 120
    frames = _noise_frames(n, rows, cols, seed=P + F)
    T = tr.transforms("walk", n, seed=P * 7 + F)
    _offline_check(frames, T, _sums(n, rows * cols, seed=P), [(0, n)], P, F, wh, tr.GLOBAL_SMOOTHING)


@pytest.mark.parametrize("kind,shards", [("large", [(0, 480)]),
                                         ("affine", [(0, 200), (200, 480)]),
                                         ("nan", [(0, 170), (170, 330), (330, 480)]),
                                         ("inf", [(0, 480)])])
def test_window_average_transform_families(kind, shards):
    """Window 150/120 (269 terms, unstaged) over large motion, affine + projective transforms and a clip with one NaN /
    inf transform (every window that holds it falls back to the identity), with shard boundaries inside windows."""
    P, F, n = 150, 120, 480
    rows, cols, wh = HALF
    T = tr.transforms("walk" if kind in ("nan", "inf") else kind, n, seed=len(kind))
    if kind in ("nan", "inf"):
        T = _with_nonfinite(T, 300, kind)
    frames = _noise_frames(n, rows, cols, seed=11)
    _offline_check(frames, T, _sums(n, rows * cols, seed=3), shards, P, F, wh, tr.GLOBAL_SMOOTHING)


@pytest.mark.parametrize("anchor,kind,geom,shards,nonfinite", [
    (0, "walk", SMALL, [(0, 1500)], None),
    (255, "large", SMALL, [(0, 700), (700, 1500)], None),
    (256, "affine", SMALL, [(0, 1500)], None),
    (257, "walk", SMALL, [(0, 500), (500, 1000), (1000, 1500)], None),
    (1000, "walk", HALF, [(0, 1500)], 1300),
])
def test_accumulated_lock_over_scan_chunks(anchor, kind, geom, shards, nonfinite):
    """ACCUMULATED_FULL_LOCK on 1500-frame clips: acc_seq_kernel's sequential prefix over 256-transform chunks from an
    anchor (lock_call - F) on and off a chunk start, every shard scanning the whole clip; window average before the
    lock call.  A NaN transform after the anchor makes every later product non-finite: decompose_h fails and the lock
    presents the identity."""
    P, F, n = 20, 12, 1500
    rows, cols, wh = geom
    T = tr.transforms(kind, n, seed=anchor + 1)
    if nonfinite is not None:
        T = _with_nonfinite(T, nonfinite, "nan")
    frames = _noise_frames(n, rows, cols, seed=anchor)
    _offline_check(frames, T, _sums(n, rows * cols, seed=anchor), shards, P, F, wh, tr.ACCUMULATED_FULL_LOCK,
                   lock_call=anchor + F)


@pytest.fixture(scope="module")
def clip_320(texture_small):
    return render_clip(texture_small, 320, 180, 400)


def test_fused_pass_deep_ring(texture_small):
    """vstab_offline_run's fused estimate + warp pass with F = 210 and chunks of B = 8 frames: the ring holds
    ceil((F-1)/B)+3 = 30 chunks.  The transforms it returns give, through the restatement, the Hs whose warp of the
    presented frame is every output, and the checksums are those of the outputs."""
    P, F, B, n = 60, 210, 8, 330
    rows, cols, wh = 192, 256, 96
    frames = np.ascontiguousarray(np.stack(render_clip(texture_small, cols, rows, n)))
    off = offline.OfflineStabilizer(P, F, wh, rows, cols, B)
    off.comm_init(0, 1)
    out = np.zeros_like(frames)
    r = off.run(n, vs.GLOBAL_SMOOTHING, 0, host_frames=frames, host_out=out, want_T=True)
    off.close()
    T = [list(t) for t in r["T"].reshape(n, 9)]
    npix = float(rows * cols)
    for c in range(n):
        want = tr.call_params(T, c, P, F, tr.GLOBAL_SMOOTHING, scale=wh / rows, npix=npix,
                              sums=frames[max(0, c - F)].reshape(-1, 3).sum(0, dtype=np.uint64).tolist())
        ref = cv2.warpPerspective(frames[want["p"]], np.reshape(want["Hs"], (3, 3)), (cols, rows), flags=cv2.INTER_LINEAR,
                                  borderMode=cv2.BORDER_CONSTANT, borderValue=tuple(float(v) for v in want["border"]))
        assert np.array_equal(out[c], ref), f"call {c}"
        assert int(r["checksums"][c]) == vs.frame_checksum(out[c]), f"call {c}"


def _stream(frames, P, F, wh, mode, lock_at, partial_fix=False):
    """Runs the streaming Stabilizer, collects per call the transform, both H taps, the border, the channel sums of the
    presented frame (vstab_read_tap: sums of frame `last_presented`) and the presentation index."""
    st = vs.Stabilizer(P, F, wh)
    if partial_fix:
        st.set_partial_lock_fix(True)
    rec = dict(T=[list(tr.I3)], Hw=[None], Hs=[None], border=[None], sums=[None], p=[0])
    for i, f in enumerate(frames):
        if i == lock_at:
            st.set_stabilization_mode(mode)
        st.stabilize_frame(f)
        if i == 0:
            continue
        rec["T"].append(st.tap(vs.TAP_T).reshape(9).tolist())
        rec["Hw"].append(st.tap(vs.TAP_H_STABILIZE).reshape(9))
        rec["Hs"].append(st.tap(vs.TAP_H_SCALED).reshape(9))
        rec["border"].append(list(st.tap(vs.TAP_BORDER)))
        rec["sums"].append(st.tap(vs.TAP_CHANNEL_SUMS).tolist())
        rec["p"].append(st.presentation_index())
    ww, whh = st.working_size()
    st.close()
    return rec, ww, whh


@pytest.mark.parametrize("wh", [180, 120])
@pytest.mark.parametrize("mode", [vs.GLOBAL_SMOOTHING, vs.ACCUMULATED_FULL_LOCK, vs.TRANSLATION_LOCK, vs.ROTATION_LOCK])
def test_streaming_long_window(clip_320, wh, mode):
    """Streaming with window 180/100 (transform ring of 283): GLOBAL_SMOOTHING throughout (279 terms, unstaged, from
    call 258 on), or GLOBAL_SMOOTHING for 130 calls and then `mode` for 270.  Window average and ACCUMULATED_FULL_LOCK
    (acc_update_kernel) bit for bit; TRANSLATION / ROTATION lock with the partial-lock fix within 1e-12 px (device
    sin / cos / atan2 against libm)."""
    P, F = 180, 100
    n = len(clip_320)
    lock_at = n if mode == vs.GLOBAL_SMOOTHING else 130
    rows, cols = clip_320[0].shape[:2]
    partial = mode in (vs.TRANSLATION_LOCK, vs.ROTATION_LOCK)
    rec, ww, whh = _stream(clip_320, P, F, wh, mode, lock_at, partial_fix=partial)
    acc = tr.accumulated(rec["T"], lock_at - F, n)
    cx, cy = float(np.float32(ww / 2.0)), float(np.float32(whh / 2.0))
    for c in range(1, n):
        m = tr.GLOBAL_SMOOTHING if c < lock_at else mode
        want = tr.call_params(rec["T"], c, P, F, m, lock_call=lock_at, acc=acc, scale=wh / rows, sums=rec["sums"][c],
                              npix=float(rows * cols), partial_fix=partial, cx=cx, cy=cy)
        assert rec["p"][c] == want["p"], c
        assert rec["border"][c] == want["border"], c
        if m in (tr.GLOBAL_SMOOTHING, tr.ACCUMULATED_FULL_LOCK):
            _assert_bits(rec["Hw"][c], want["Hw"], f"call {c} H_stabilize")
            _assert_bits(rec["Hs"][c], want["Hs"], f"call {c} H_scaled")
        else:
            assert tr.corner_diff(rec["Hs"][c], want["Hs"], cols, rows) <= 1e-12, c
            assert tr.corner_diff(rec["Hw"][c], want["Hw"], ww, whh) <= 1e-12, c


def test_oracle_long_window(clip_320):
    """The reference pipeline against the engine with window 150/120 (269 terms, past the shared-memory stage),
    300 frames of 320x180 at working height 180, under the bars of the other oracle runs."""
    from test_gpu_pipeline import FRAC_GT1, H_ACHIEVED_PX, MAX_Q5_STEP, _run_both
    s = _run_both(clip_320[:300], 150, 120, 180)
    assert s["corners_differ"] == 0 and s["status"] == 0 and s["lk"] == 0.0
    assert s["h"] <= H_ACHIEVED_PX
    assert s["frac_gt1"] <= FRAC_GT1 and s["pix"] <= MAX_Q5_STEP
