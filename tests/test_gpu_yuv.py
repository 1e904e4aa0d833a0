"""YUV 4:2:0 frames on the GPU: the K15 kernels are byte-identical to cv2, and every entry point that takes or returns
NV12 / I420 frames returns, call by call, to_yuv(the BGR path's output on from_yuv(input)) -- streaming (host and device
buffers, every mode family, future 0 / 1 / 9, mixed with BGR calls), vstab_offline_run_host, vstab_offline_run (host and
device sources and sinks, fused and two-pass) and the file front end."""
import os
import subprocess

import numpy as np
import pytest

import vstab_b200 as vs
from vstab_b200 import offline
from oracle import synth
from yuv_ref import I420, NV12, bgr_to_yuv420, join_planes, split_planes, yuv420_to_bgr

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
cv2 = pytest.importorskip("cv2")


def _clip_yuv(tex, W, H, n, fmt):
    """a rendered clip as packed 4:2:0 frames (what a decoder would hand over)"""
    from conftest import render_clip
    return [bgr_to_yuv420(f, fmt) for f in render_clip(tex, W, H, n)]


def _place(planes, fmt, steps, offsets, total):
    """a host frame buffer of `total` bytes (0xEE elsewhere) holding the planes at the given offsets / steps"""
    buf = np.full(total, 0xEE, np.uint8)
    Y, U, V = planes
    rows, cols = Y.shape
    chroma = [np.stack([U, V], -1).reshape(rows // 2, cols)] if fmt == NV12 else [U, V]
    for k, p in enumerate([Y] + chroma):
        for r in range(p.shape[0]):
            buf[offsets[k] + r * steps[k]: offsets[k] + r * steps[k] + p.shape[1]] = p[r]
    return buf, vs.YuvLayout.make(fmt, offsets, steps)


def _layouts(fmt, rows, cols):
    """packed; padded steps with odd padding (byte path); planes apart with gaps (offsets not adjacent), 8-byte aligned"""
    cw = cols if fmt == NV12 else cols // 2
    yield "packed", None
    y_st, c_st = cols + 3, cw + 5
    off = [1, 1 + y_st * rows + 7]
    if fmt == I420:
        off.append(off[1] + c_st * (rows // 2) + 11)
    yield "padded", (([y_st] + [c_st] * (2 if fmt == I420 else 1)), off)
    y_st, c_st = cols + 64, cw + 32
    y_st, c_st = (y_st + 7) // 8 * 8, (c_st + 7) // 8 * 8
    off = [4096, 4096 + y_st * rows + 8192]
    if fmt == I420:
        off.append(off[1] + c_st * (rows // 2) + 4096)
    yield "apart", (([y_st] + [c_st] * (2 if fmt == I420 else 1)), off)


# ---------------------------------------------------------------- 1. kernels
@pytest.mark.parametrize("fmt", [NV12, I420])
@pytest.mark.parametrize("rows,cols", [(1080, 1920), (250, 334), (12, 12)])
def test_kernels_equal_cv2(fmt, rows, cols):
    rng = np.random.default_rng(rows + cols + fmt)
    yuv = rng.integers(0, 256, (rows * 3 // 2, cols), dtype=np.uint8)
    if fmt == I420:
        want_bgr = cv2.cvtColor(yuv, cv2.COLOR_YUV2BGR_I420)
    else:
        want_bgr = cv2.cvtColor(yuv, cv2.COLOR_YUV2BGR_NV12)
    bgr = rng.integers(0, 256, (rows, cols, 3), dtype=np.uint8)
    i420 = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)
    want_yuv = i420 if fmt == I420 else join_planes(*split_planes(i420, I420), NV12)
    for name, spec in _layouts(fmt, rows, cols):
        if spec is None:
            assert np.array_equal(vs.k_yuv_to_bgr(yuv, fmt), want_bgr), name
            assert np.array_equal(vs.k_bgr_to_yuv(bgr, fmt), want_yuv), name
            continue
        steps, offs = spec
        total = offs[-1] + steps[-1] * (rows // 2) + 64
        src, L = _place(split_planes(yuv, fmt), fmt, steps, offs, total)
        assert np.array_equal(vs.k_yuv_to_bgr(src, L, rows, cols), want_bgr), name
        want_buf, _ = _place(split_planes(want_yuv, fmt), fmt, steps, offs, total)
        out = np.full(total, 0xEE, np.uint8)
        vs.k_bgr_to_yuv(bgr, L, out)
        assert np.array_equal(out, want_buf), name            # the planes' bytes, and nothing between them


# ---------------------------------------------------------------- 2. streaming
def _bgr_streaming(frames_bgr, P, F, wh, setup, events):
    st = vs.Stabilizer(P, F, wh)
    setup(st)
    outs = []
    for i, f in enumerate(frames_bgr):
        if i in events:
            events[i](st)
        outs.append(st.stabilize_frame(f))
    st.close()
    return outs


def _dev_layout(fmt, rows, cols, pad):
    """device frame in separate allocations (an NVDEC-like pitched surface): Y and chroma tensors, base = the lower one"""
    cw = cols if fmt == NV12 else cols // 2
    ys, cs = cols + pad, cw + pad
    y = torch.zeros((rows, ys), dtype=torch.uint8, device="cuda")
    cp = [torch.zeros((rows // 2, cs), dtype=torch.uint8, device="cuda") for _ in range(1 if fmt == NV12 else 2)]
    ptrs = [y.data_ptr()] + [c.data_ptr() for c in cp]
    base = min(ptrs)
    L = vs.YuvLayout.make(fmt, [p - base for p in ptrs], [ys] + [cs] * len(cp))
    return [y] + cp, base, L


def _dev_write(tensors, frame, fmt):
    Y, U, V = split_planes(frame, fmt)
    rows, cols = Y.shape
    chroma = [np.stack([U, V], -1).reshape(rows // 2, cols)] if fmt == NV12 else [U, V]
    for t, p in zip(tensors, [Y] + chroma):
        t[:, :p.shape[1]].copy_(torch.from_numpy(np.ascontiguousarray(p)))


def _dev_read(tensors, fmt, rows, cols):
    ps = [t.cpu().numpy() for t in tensors]
    Y = ps[0][:, :cols]
    if fmt == NV12:
        uv = ps[1][:, :cols].reshape(rows // 2, cols // 2, 2)
        return join_planes(Y, uv[..., 0], uv[..., 1], NV12)
    return join_planes(Y, ps[1][:, :cols // 2], ps[2][:, :cols // 2], I420)


CASES = [  # (name, P, F, wh, W, H, in fmt, out fmt, device)
    ("global", 5, 0, 120, 320, 240, NV12, I420, False),
    ("global", 5, 1, 120, 320, 240, I420, NV12, True),
    ("global", 4, 9, 120, 320, 240, NV12, NV12, False),
    ("lock", 4, 9, 120, 320, 240, I420, NV12, False),
    ("lock", 5, 1, 120, 320, 240, NV12, I420, True),
    ("lock", 5, 0, 120, 320, 240, I420, I420, False),
    ("orb", 5, 3, 360, 640, 360, NV12, I420, False),
    ("orb", 5, 1, 360, 640, 360, I420, NV12, True),
    ("trail", 4, 9, 120, 320, 240, I420, I420, False),
    ("trail", 5, 1, 120, 320, 240, NV12, NV12, True),
]


@pytest.mark.parametrize("name,P,F,wh,W,H,fin,fout,device", CASES)
def test_streaming_yuv_equals_bgr_path(texture_small, name, P, F, wh, W, H, fin, fout, device):
    n = 22
    lock_at = 12
    frames = _clip_yuv(texture_small, W, H, n, fin)
    setup = (lambda st: st.set_trail(True)) if name == "trail" else (lambda st: None)
    mode = {"lock": vs.ACCUMULATED_FULL_LOCK, "orb": vs.ORB_FULL_LOCK}.get(name)
    events = {lock_at: (lambda st: st.set_stabilization_mode(mode))} if mode is not None else {}
    want = [bgr_to_yuv420(o, fout) for o in _bgr_streaming([yuv420_to_bgr(f, fin) for f in frames], P, F, wh, setup, events)]
    st = vs.Stabilizer(P, F, wh)
    setup(st)
    if device:
        tin, bin_, Lin = _dev_layout(fin, H, W, 24)
        tout, bout, Lout = _dev_layout(fout, H, W, 40)
    for i, f in enumerate(frames):
        if i in events:
            events[i](st)
        if device:
            _dev_write(tin, f, fin)
            torch.cuda.synchronize()
            st.stabilize_frame_yuv_ptr(bin_, Lin, H, W, bout, Lout, device=True)
            st.synchronize()
            got = _dev_read(tout, fout, H, W)
        else:
            got = st.stabilize_frame_yuv(f, fin, out_fmt=fout)
        assert np.array_equal(got, want[i]), f"{name} call {i}"
    st.close()


def test_streaming_yuv_against_the_oracle_with_cv2_conversions(texture_small):
    """GLOBAL_SMOOTHING on I420 frames == cv2 BGR2YUV_I420(oracle stabilizeFrame(cv2 YUV2BGR_I420(frame)))"""
    from oracle import stabilizer_ref as sr
    W, H, n, P, F, wh = 256, 192, 12, 4, 3, 96
    frames = _clip_yuv(texture_small, W, H, n, I420)
    ref = sr.StabilizerRef(P, F, wh)
    st = vs.Stabilizer(P, F, wh)
    for i, f in enumerate(frames):
        want = cv2.cvtColor(ref.stabilize_frame(cv2.cvtColor(f, cv2.COLOR_YUV2BGR_I420)), cv2.COLOR_BGR2YUV_I420)
        got = st.stabilize_frame_yuv(f, vs.PIX_I420)
        d = np.abs(got.astype(int) - want)
        assert d.max() <= 1, (i, int(d.max()))                # the BGR path's bar against the oracle (smoke(): 1 LSB)
    st.close()


def test_streaming_mixed_bgr_and_yuv_calls(texture_small):
    """BGR and NV12 calls alternate on one instance: the window holds BGR either way, so the outputs are the all-BGR ones"""
    W, H, n, P, F, wh = 320, 240, 16, 4, 3, 120
    frames = _clip_yuv(texture_small, W, H, n, NV12)
    bgr = [yuv420_to_bgr(f, NV12) for f in frames]
    want = _bgr_streaming(bgr, P, F, wh, lambda st: None, {7: lambda st: st.set_stabilization_mode(vs.ACCUMULATED_FULL_LOCK)})
    st = vs.Stabilizer(P, F, wh)
    for i in range(n):
        if i == 7:
            st.set_stabilization_mode(vs.ACCUMULATED_FULL_LOCK)
        if i % 2:
            assert np.array_equal(st.stabilize_frame_yuv(frames[i], vs.PIX_NV12), bgr_to_yuv420(want[i], NV12)), i
        else:
            assert np.array_equal(st.stabilize_frame(bgr[i]), want[i]), i
    st.close()


def test_streaming_yuv_argument_errors(texture_small):
    st = vs.Stabilizer(4, 3, 120)
    with pytest.raises(ValueError):
        st.stabilize_frame_yuv(np.zeros((360, 319), np.uint8), vs.PIX_NV12)        # odd width
    with pytest.raises(ValueError):
        st.stabilize_frame_yuv(np.zeros((15, 10), np.uint8), vs.PIX_NV12)          # 10 rows: the reference's size check
    f = _clip_yuv(texture_small, 320, 240, 1, NV12)[0]
    st.stabilize_frame_yuv(f, vs.PIX_NV12)
    with pytest.raises(ValueError, match="size has changed"):
        st.stabilize_frame_yuv(np.zeros((240, 320), np.uint8), vs.PIX_NV12)
    with pytest.raises(ValueError):
        st.stabilize_frame_yuv(f, 7)
    st.close()


# ---------------------------------------------------------------- 3. run_host
@pytest.mark.parametrize("fin,fout,lock_at", [(NV12, NV12, None), (I420, NV12, 9), (NV12, I420, None)])
def test_run_host_yuv_equals_streaming_yuv(texture_small, fin, fout, lock_at):
    """chunks of 7 frames over 30 (the last chunk is short); the second run reuses the instance's staging buffers"""
    W, H, wh, P, F, n = 480, 270, 135, 6, 4, 30
    frames = _clip_yuv(texture_small, W, H, n, fin)
    st = vs.Stabilizer(P, F, wh)
    want = []
    for i, f in enumerate(frames):
        if lock_at is not None and i == lock_at:
            st.set_stabilization_mode(vs.ACCUMULATED_FULL_LOCK)
        want.append(st.stabilize_frame_yuv(f, fin, out_fmt=fout))
    st.close()
    clip = np.ascontiguousarray(np.stack(frames))
    out = np.zeros_like(clip)
    off = offline.OfflineStabilizer(P, F, wh, H, W, 7)
    off.set_yuv(fin, fout)
    mode = vs.GLOBAL_SMOOTHING if lock_at is None else vs.ACCUMULATED_FULL_LOCK
    for _ in range(2):
        off.run_host(clip.ctypes.data, clip.strides[0], 0, n, mode, lock_at or 0, out.ctypes.data, out.strides[0], 0)
        for c in range(n):
            assert np.array_equal(out[c], want[c]), c
        out[:] = 0
    off.set_yuv(None, None)                                   # back to BGR on the same instance
    bgr = np.ascontiguousarray(np.stack([yuv420_to_bgr(f, fin) for f in frames]))
    ob = np.zeros_like(bgr)
    off.run_host(bgr.ctypes.data, bgr.strides[0], bgr.strides[1], n, mode, lock_at or 0, ob.ctypes.data, ob.strides[0], ob.strides[1])
    for c in range(n):
        assert np.array_equal(bgr_to_yuv420(ob[c], fout), want[c]), c
    off.close()


# ---------------------------------------------------------------- 4. vstab_offline_run
def _bgr_job(off, n, mode, lock_at, frames_bgr):
    out = np.zeros((n,) + frames_bgr.shape[1:], np.uint8)
    r = off.run(n, mode, lock_at, host_frames=frames_bgr, host_out=out, want_T=True)
    return r, out


@pytest.mark.parametrize("mode,lock_at,B", [(vs.GLOBAL_SMOOTHING, 0, 2), (vs.GLOBAL_SMOOTHING, 0, 3), (vs.GLOBAL_SMOOTHING, 0, 16),
                                            (vs.GLOBAL_SMOOTHING, 0, 64), (vs.ACCUMULATED_FULL_LOCK, 11, 5)])
def test_offline_run_yuv_equals_bgr_job(texture_small, mode, lock_at, B):
    """HOST and DEVICE YUV sources into host_out and d_out YUV sinks: checksums and T_all are those of the BGR job on the
    converted clip, outputs are its outputs converted.  GLOBAL_SMOOTHING takes the fused pass (ring shapes of
    test_offline_run_fused_pass_ring_shapes), ACCUMULATED_FULL_LOCK the two passes."""
    W, H, wh, n, P, F = 480, 270, 135, 41, 7, 9
    fin, fout = (NV12, I420) if B % 2 else (I420, NV12)
    frames = np.ascontiguousarray(np.stack(_clip_yuv(texture_small, W, H, n, fin)))
    bgr = np.ascontiguousarray(np.stack([yuv420_to_bgr(f, fin) for f in frames]))
    off = offline.OfflineStabilizer(P, F, wh, H, W, B)
    off.comm_init(0, 1)
    want_r, want_out = _bgr_job(off, n, mode, lock_at, bgr)
    want = np.stack([bgr_to_yuv420(o, fout) for o in want_out])
    off.set_yuv(fin, fout)
    got_host = np.zeros_like(want)
    r1 = off.run(n, mode, lock_at, host_frames=frames, host_out=got_host, want_T=True)
    dev_in = torch.from_numpy(frames).cuda()
    got_dev = torch.zeros((n, H * 3 // 2, W), dtype=torch.uint8, device="cuda")
    r2 = off.run(n, mode, lock_at, device_frames=dev_in, device_out=got_dev, want_T=True)
    got_mix = torch.zeros_like(got_dev)
    r3 = off.run(n, mode, lock_at, host_frames=frames, device_out=got_mix, want_T=True)
    off.close()
    for r in (r1, r2, r3):
        assert np.array_equal(r["checksums"], want_r["checksums"])
        assert np.array_equal(r["T"], want_r["T"])
    assert np.array_equal(got_host, want)
    assert np.array_equal(got_dev.cpu().numpy(), want)
    assert np.array_equal(got_mix.cpu().numpy(), want)


# ---------------------------------------------------------------- 5. file front end
def test_file_front_end_nv12_equals_streaming_yuv_api(tmp_path, texture_small):
    W, H, n, P, F, wh = 320, 240, 14, 4, 3, 120
    frames = _clip_yuv(texture_small, W, H, n, NV12)
    clip = tmp_path / "in.nv12"
    clip.write_bytes(b"".join(f.tobytes() for f in frames))
    out = tmp_path / "out.yuv"
    exe = os.path.join(os.path.dirname(os.path.dirname(vs.LIB_PATH)), "bin", "vstab_file")
    cmd = [exe, "--file", str(clip), "--width", str(W), "--height", str(H), "--out", str(out), "--past-window", str(P),
           "--future-window", str(F), "--working-height", str(wh), "--mode", "lock", "--mode-at", "5",
           "--pix-fmt", "nv12", "--out-pix-fmt", "yuv420p"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    st = vs.Stabilizer(P, F, wh)
    got = np.frombuffer(out.read_bytes(), np.uint8).reshape(n, H * 3 // 2, W)
    for i, f in enumerate(frames):
        if i == 5:
            st.set_stabilization_mode(vs.ACCUMULATED_FULL_LOCK)
        assert np.array_equal(got[i], st.stabilize_frame_yuv(f, vs.PIX_NV12, out_fmt=vs.PIX_I420)), i
    st.close()
