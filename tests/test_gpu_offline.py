"""T4: the offline (batched, frame-sharded) runner reproduces the streaming Stabilizer for every
call index (SURVEY.md Appendix C), including shard boundaries and the ACCUMULATED_FULL_LOCK
anchor; and the device simulator (K13) renders the same bytes as the CPU restatement of
CameraEngine::renderFrame."""
import numpy as np
import pytest

import vstab_b200 as vs
from vstab_b200 import offline
from oracle import camera_engine_ref as ce
from oracle import synth

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def _dev_clip(tex_np, W, H, n, start=0):
    tex = torch.from_numpy(tex_np).cuda()
    path = synth.camera_path(start + n)[start:]
    out = torch.empty((n, H, W, 3), dtype=torch.uint8, device="cuda")
    offline.render_frames(tex, path, H, W, synth.focal_for_width(W), out)
    return out, path


@pytest.mark.parametrize("W,H", [(640, 360), (1280, 720), (333, 250)])
def test_render_matches_camera_engine(texture_small, W, H):
    """K13 == CameraEngine::renderFrame (src/camera_engine.cpp:73-172): identical texel choices."""
    frames, path = _dev_clip(texture_small, W, H, 3, start=5)
    for i in range(3):
        ref = ce.render_frame(texture_small, path[i], W, H, synth.focal_for_width(W))
        assert np.array_equal(frames[i].cpu().numpy(), ref)


@pytest.mark.parametrize("rows,cols", [(384, 512), (512, 300)])
def test_render_non_square_texture(texture_small, rows, cols):
    """tileHeight = 1 / aspect != 1 (camera_engine.cpp:81-88): worldY / tileHeight is a real division per pixel; 7 frames,
    so that the per-thread frame loop (4 frames per thread) has a partial last group."""
    W, H, n = 640, 360, 7
    tex_np = np.ascontiguousarray(texture_small[:rows, :cols])
    frames, path = _dev_clip(tex_np, W, H, n, start=3)
    got = frames.cpu().numpy()
    for i in range(n):
        ref = ce.render_frame(tex_np, path[i], W, H, synth.focal_for_width(W))
        assert np.array_equal(got[i], ref), i
    # the job's renderer (ray table + BGRX texture) against the stand-alone one (rays computed, BGR texture)
    off = offline.OfflineStabilizer(3, 2, 180, H, W, 3)
    off.comm_init(0, 1)
    a = off.run(n, vs.GLOBAL_SMOOTHING, 0, texture=torch.from_numpy(tex_np).cuda(), poses=path, focal=synth.focal_for_width(W))
    b = off.run(n, vs.GLOBAL_SMOOTHING, 0, host_frames=got)
    off.close()
    assert np.array_equal(a["checksums"], b["checksums"])


def test_render_sky_and_tilted_pose(texture_small):
    """A tilted camera sees the horizon: sky colour above it (camera_engine.cpp:119), floor below."""
    W, H = 320, 240
    poses = np.array([[0.5, -0.3, 0.7, 5.0, 80.0, 170.0], [0.2, 0.1, 1.5, -30.0, 95.0, 182.0]])
    tex = torch.from_numpy(texture_small).cuda()
    out = torch.empty((2, H, W, 3), dtype=torch.uint8, device="cuda")
    offline.render_frames(tex, poses, H, W, 250.0, out)
    for i in range(2):
        ref = ce.render_frame(texture_small, poses[i], W, H, 250.0)
        got = out[i].cpu().numpy()
        assert (ref == np.array([230, 216, 173], np.uint8)).all(axis=2).any()      # some sky is visible
        assert (got != ref).any(axis=2).mean() <= 1e-4                              # libm vs CUDA trig in R: <= a few texels


def _streaming(frames_np, P, F, wh, lock_at):
    st = vs.Stabilizer(P, F, wh)
    outs, Hs = [], []
    for i, f in enumerate(frames_np):
        if lock_at is not None and i == lock_at:
            st.set_stabilization_mode(vs.ACCUMULATED_FULL_LOCK)
        outs.append(st.stabilize_frame(f))
        Hs.append(st.tap(vs.TAP_H_SCALED) if i else np.eye(3))
    st.close()
    return outs, Hs


def _offline(frames, shards, P, F, wh, mode, lock_call, batch):
    """Runs every shard on this one GPU (ranks emulated one after the other, no collective: the
    gather is a torch.cat), returns outputs by call index."""
    n_total, H, W = frames.shape[0], frames.shape[1], frames.shape[2]
    T_parts, sums_parts, runners = [], [], []
    for (first, last) in shards:
        off = offline.OfflineStabilizer(P, F, wh, H, W, batch)
        T = torch.zeros((last - first, 9), dtype=torch.float64, device="cuda")
        sums = torch.zeros((last - first, 3), dtype=torch.int64, device="cuda")
        off.estimate(frames[first:last], first, frames[first - 1] if first else None, T, sums)
        off.synchronize()
        T_parts.append(T); sums_parts.append(sums); runners.append(off)
    T_all = torch.cat(T_parts, 0)
    outs, Hs = {}, {}
    for (first, last), sums, off in zip(shards, sums_parts, runners):
        c0, c1 = offline.calls_of_shard(first, last, n_total, F)
        if c1 <= c0:
            continue
        out = torch.empty((c1 - c0, H, W, 3), dtype=torch.uint8, device="cuda")
        off.prepare(T_all, mode, lock_call)
        done = 0
        while done < c1 - c0:                      # batch by batch so read_h sees each launch
            m = min(batch, c1 - c0 - done)
            off.render(frames[first:last], first, c0 + done, m, T_all, mode, lock_call, sums, out[done:])
            hs = off.read_h(m)
            for j in range(m):
                Hs[c0 + done + j] = hs[j]
            done += m
        off.synchronize()
        o = out.cpu().numpy()
        for j in range(c1 - c0):
            outs[c0 + j] = o[j]
        off.close()
    return outs, Hs


@pytest.mark.parametrize("lock_at", [None, 9])
@pytest.mark.parametrize("shards", [[(0, 30)], [(0, 15), (15, 30)], [(0, 7), (7, 19), (19, 30)]])
def test_offline_equals_streaming(texture_small, lock_at, shards):
    W, H, wh, P, F = 480, 270, 135, 6, 4
    frames, _ = _dev_clip(texture_small, W, H, 30)
    f_np = frames.cpu().numpy()
    want, want_H = _streaming(f_np, P, F, wh, lock_at)
    mode = vs.GLOBAL_SMOOTHING if lock_at is None else vs.ACCUMULATED_FULL_LOCK
    got, got_H = _offline(frames, shards, P, F, wh, mode, lock_at or 0, batch=7)
    assert sorted(got) == list(range(30))                 # every call index produced exactly once
    for c in range(30):
        if c == 0:
            # call 0 returns the input frame (stabilizer.cpp:1181); offline renders it through the
            # identity warp of frame 0 -- same bytes
            assert np.array_equal(got[0], f_np[0])
            continue
        assert np.array_equal(got_H[c], want_H[c]), c      # same kernels, same order: bit-identical H
        assert np.array_equal(got[c], want[c]), c


@pytest.mark.parametrize("mode,lock_at,F", [pytest.param(vs.GLOBAL_SMOOTHING, None, 4, id="None"),
                                            pytest.param(vs.ACCUMULATED_FULL_LOCK, 9, 4, id="9"),
                                            pytest.param(vs.ACCUMULATED_FULL_LOCK, 9, 0, id="future0-9"),
                                            pytest.param(vs.ORB_FULL_LOCK, 9, 4, id="orb-9")])
def test_run_host_equals_streaming(texture_small, mode, lock_at, F):
    """vstab_offline_run_host (vstab_offline_run's job on one GPU: uploads / estimation / warps / downloads pipelined over
    host buffers) returns exactly the frames the streaming calls return: with future 0 (a call presents the frame it
    receives), and in ORB lock (at the size of the feature-lock test below)."""
    W, H, wh = (640, 360, 360) if mode == vs.ORB_FULL_LOCK else (480, 270, 135)
    P = 6
    frames, _ = _dev_clip(texture_small, W, H, 30)
    f_np = np.ascontiguousarray(frames.cpu().numpy())
    want = _streaming_mode(f_np, P, F, wh, mode, lock_at)
    out = np.zeros_like(f_np)
    off = offline.OfflineStabilizer(P, F, wh, H, W, 7)
    for _ in range(2):                    # second run reuses the instance's chunk ring and output chunks
        off.run_host(f_np.ctypes.data, f_np.strides[0], f_np.strides[1], 30, mode, lock_at or 0,
                     out.ctypes.data, out.strides[0], out.strides[1])
        for c in range(30):
            assert np.array_equal(out[c], want[c]), c
        out[:] = 0
    off.close()


@pytest.mark.parametrize("mode", [vs.ORB_FULL_LOCK, vs.SIFT_FULL_LOCK])
@pytest.mark.parametrize("shards", [[(0, 20)], [(0, 9), (9, 20)]])
def test_offline_feature_lock_equals_streaming(texture_small, mode, shards):
    """ORB / SIFT registration offline (reference broadcast + independent per-frame registration + gathered
    {H, valid} + carry scan) == the streaming calls, bit for bit, across a shard boundary."""
    W, H, wh, P, F, lock_at, n_total = 640, 360, 360, 5, 3, 6, 20
    frames, _ = _dev_clip(texture_small, W, H, n_total)
    f_np = frames.cpu().numpy()
    st = vs.Stabilizer(P, F, wh)
    want, want_H = [], []
    for i, f in enumerate(f_np):
        if i == lock_at:
            st.set_stabilization_mode(mode)
        want.append(st.stabilize_frame(f))
        want_H.append(st.tap(vs.TAP_H_SCALED) if i else np.eye(3))
    st.close()
    anchor = max(0, lock_at - F)
    runners, T_parts, sums_parts, reg_parts = [], [], [], []
    pack = None
    for (first, last) in shards:
        off = offline.OfflineStabilizer(P, F, wh, H, W, 32)
        T = torch.zeros((last - first, 9), dtype=torch.float64, device="cuda")
        sums = torch.zeros((last - first, 3), dtype=torch.int64, device="cuda")
        off.estimate(frames[first:last], first, frames[first - 1] if first else None, T, sums)
        if first <= anchor < last:
            off.capture_reference(frames[anchor], mode)
            pack = off.export_reference()
        runners.append(off); T_parts.append(T); sums_parts.append(sums)
    for (first, last), off in zip(shards, runners):
        if not (first <= anchor < last):
            off.import_reference(pack, mode)                  # the "broadcast"
        reg = torch.zeros((last - first, 10), dtype=torch.float64, device="cuda")
        off.register(frames[first:last], reg)
        off.synchronize()
        reg_parts.append(reg)
    T_all, reg_all = torch.cat(T_parts, 0), torch.cat(reg_parts, 0)     # the "all-gather"
    assert float(reg_all[anchor + 1:, 9].min()) == 1.0
    for (first, last), sums, off in zip(shards, sums_parts, runners):
        c0, c1 = offline.calls_of_shard(first, last, n_total, F)
        out = torch.empty((c1 - c0, H, W, 3), dtype=torch.uint8, device="cuda")
        off.set_registrations(reg_all)
        off.prepare(T_all, mode, lock_at)
        off.render(frames[first:last], first, c0, c1 - c0, T_all, mode, lock_at, sums, out)
        hs = off.read_h(c1 - c0)
        o = out.cpu().numpy()
        for j in range(c1 - c0):
            c = c0 + j
            if c:
                assert np.array_equal(hs[j], want_H[c]), c
            assert np.array_equal(o[j], want[c]), c
        off.close()


# ---------------------------------------------------------------- vstab_offline_run (the sharded job behind one call)
def _streaming_mode(frames_np, P, F, wh, mode, lock_at):
    st = vs.Stabilizer(P, F, wh)
    outs = []
    for i, f in enumerate(frames_np):
        if lock_at is not None and i == lock_at:
            st.set_stabilization_mode(mode)
        outs.append(st.stabilize_frame(f))
    st.close()
    return outs


@pytest.mark.parametrize("mode,lock_at,W,H,wh", [(vs.GLOBAL_SMOOTHING, None, 640, 360, 180),
                                                 (vs.ACCUMULATED_FULL_LOCK, 9, 640, 360, 180),
                                                 (vs.ORB_FULL_LOCK, 8, 640, 360, 360)])
def test_offline_run_world_of_one_equals_streaming(texture_small, mode, lock_at, W, H, wh):
    """vstab_offline_run with the simulator source (two passes, chunks of 5 frames resident at a time) and with the
    host source gives, call by call, the bytes of the streaming Stabilizer -- and the checksum the warp kernel fuses
    equals vstab_frame_checksum of those bytes."""
    n, P, F, B = 23, 6, 4, 5
    frames, path = _dev_clip(texture_small, W, H, n)
    frames_np = frames.cpu().numpy()
    want = _streaming_mode(frames_np, P, F, wh, mode, lock_at)
    tex = torch.from_numpy(texture_small).cuda()
    off = offline.OfflineStabilizer(P, F, wh, H, W, B)
    off.comm_init(0, 1)
    host_out = np.zeros((n, H, W, 3), np.uint8)
    r = off.run(n, mode, lock_at or 0, texture=tex, poses=path, focal=synth.focal_for_width(W), host_out=host_out)
    assert (r["first"], r["last"], r["call_first"], r["call_last"]) == (0, n, 0, n)
    for c in range(n):
        assert np.array_equal(host_out[c], want[c]), f"call {c}"
        assert int(r["checksums"][c]) == vs.frame_checksum(want[c])
    # host source, odd-width frames take the non-vector store / checksum path elsewhere; here: same clip from host memory
    host_out2 = np.zeros_like(host_out)
    r2 = off.run(n, mode, lock_at or 0, host_frames=frames_np, host_out=host_out2, want_T=True)
    assert np.array_equal(host_out2, host_out) and np.array_equal(r2["checksums"], r["checksums"])
    assert r2["T"].shape == (n, 3, 3) and r2["frames"] == n and r2["calls"] == n
    off.close()


def test_frame_checksum_odd_width_and_c_twin(texture_small):
    """Checksum of a warp output whose width is not a multiple of 4 (scalar store path, zero-padded last group)."""
    import ctypes as C
    W, H = 333, 250
    frames, path = _dev_clip(texture_small, W, H, 9)
    off = offline.OfflineStabilizer(3, 2, 100, H, W, 4)
    off.comm_init(0, 1)
    out = np.zeros((9, H, W, 3), np.uint8)
    r = off.run(9, vs.GLOBAL_SMOOTHING, 0, host_frames=frames.cpu().numpy(), host_out=out)
    lib = vs.load_library()
    for c in range(9):
        assert int(r["checksums"][c]) == vs.frame_checksum(out[c])
        assert vs.frame_checksum(out[c]) == lib.vstab_frame_checksum(out[c].ctypes.data_as(C.c_void_p), H, W, W * 3)
    off.close()


def test_offline_run_resident_source_equals_simulator_source(texture_small):
    """VSTAB_SRC_DEVICE (shard resident in HBM, device sink) == VSTAB_SRC_SIMULATOR for the same clip."""
    W, H, n = 640, 360, 19
    frames, path = _dev_clip(texture_small, W, H, n)
    tex = torch.from_numpy(texture_small).cuda()
    off = offline.OfflineStabilizer(5, 3, 180, H, W, 4)
    off.comm_init(0, 1)
    a = off.run(n, vs.ACCUMULATED_FULL_LOCK, 7, texture=tex, poses=path, focal=synth.focal_for_width(W))
    out = torch.zeros((n, H, W, 3), dtype=torch.uint8, device="cuda")
    b = off.run(n, vs.ACCUMULATED_FULL_LOCK, 7, device_frames=frames, device_out=out)
    assert np.array_equal(a["checksums"], b["checksums"])
    got = out.cpu().numpy()
    for c in range(n):
        assert int(b["checksums"][c]) == vs.frame_checksum(got[c])
    off.close()


@pytest.mark.parametrize("B", [2, 3, 16, 64])
def test_offline_run_fused_pass_ring_shapes(texture_small, B):
    """GLOBAL_SMOOTHING from a staged source is one fused pass over a ring of ceil((F-1)/B)+3 chunks (vstab_offline_run):
    every ring depth (B < F-1: several chunks of lag; B > clip: one chunk) returns the streaming calls' bytes, from the
    simulator source and from host frames, and equals the two-pass schedule (VSTAB_SRC_DEVICE never fuses)."""
    W, H, wh, n, P, F = 480, 270, 135, 41, 7, 9
    frames, path = _dev_clip(texture_small, W, H, n)
    frames_np = frames.cpu().numpy()
    want = _streaming_mode(frames_np, P, F, wh, vs.GLOBAL_SMOOTHING, None)
    tex = torch.from_numpy(texture_small).cuda()
    off = offline.OfflineStabilizer(P, F, wh, H, W, B)
    off.comm_init(0, 1)
    out_sim = np.zeros((n, H, W, 3), np.uint8)
    r = off.run(n, vs.GLOBAL_SMOOTHING, 0, texture=tex, poses=path, focal=synth.focal_for_width(W), host_out=out_sim)
    out_host = np.zeros_like(out_sim)
    r2 = off.run(n, vs.GLOBAL_SMOOTHING, 0, host_frames=frames_np, host_out=out_host, want_T=True)
    out_dev = torch.zeros((n, H, W, 3), dtype=torch.uint8, device="cuda")
    r3 = off.run(n, vs.GLOBAL_SMOOTHING, 0, device_frames=frames, device_out=out_dev, want_T=True)
    off.close()
    for c in range(n):
        assert np.array_equal(out_sim[c], want[c]), f"simulator source, call {c}"
        assert np.array_equal(out_host[c], want[c]), f"host source, call {c}"
    assert np.array_equal(r["checksums"], r2["checksums"]) and np.array_equal(r["checksums"], r3["checksums"])
    assert np.array_equal(r2["T"], r3["T"])
    assert np.array_equal(out_dev.cpu().numpy(), out_host)
