"""BGR frames in caller layouts that the other tests do not reach: every entry point returns the bytes of the streaming
calls on packed frames, and no byte of the caller's buffers outside the frames' pixels is read into a frame or written --
rows padded by an odd number of bytes, frames a library frame (g.frame_bytes) apart with a gap after each frame's pixels,
and tightly packed frames that move in one copy per run."""
import numpy as np
import pytest

import vstab_b200 as vs
from vstab_b200 import offline
from oracle import synth

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

W, H, WH, P, F, N, B = 480, 270, 135, 6, 4, 30, 7
SENTINEL = 0xEE
MODES = [(vs.GLOBAL_SMOOTHING, 0), (vs.ACCUMULATED_FULL_LOCK, 11)]     # window average, then the prefix rescanned per chunk


def _clip(tex_np, w, h, n):
    tex = torch.from_numpy(tex_np).cuda()
    out = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda")
    offline.render_frames(tex, synth.camera_path(n), h, w, synth.focal_for_width(w), out)
    return np.ascontiguousarray(out.cpu().numpy())


def _streaming(frames, mode, lock_at, wh=WH):
    st = vs.Stabilizer(P, F, wh)
    outs = []
    for i, f in enumerate(frames):
        if mode != vs.GLOBAL_SMOOTHING and i == lock_at:
            st.set_stabilization_mode(mode)
        outs.append(st.stabilize_frame(f))
    st.close()
    return np.stack(outs)


class Strided:
    """n frames of h x w BGR pixels in one flat buffer: rows `step` bytes apart, frames `stride` apart, `tail` bytes after
    the last frame's stride; every other byte holds SENTINEL"""

    def __init__(self, n, h, w, step, stride, tail=64):
        self.shape, self.strides = (n, h, w, 3), (stride, step, 3, 1)
        self.buf = np.full(stride * n + tail, SENTINEL, np.uint8)
        self.frames = np.lib.stride_tricks.as_strided(self.buf, self.shape, self.strides)
        pixels = np.zeros(self.buf.shape, bool)
        np.lib.stride_tricks.as_strided(pixels, self.shape, self.strides)[...] = True
        self.outside = ~pixels

    def untouched(self, buf=None):
        return bool(np.all((self.buf if buf is None else buf)[self.outside] == SENTINEL))

    def device(self):
        d = torch.from_numpy(self.buf).cuda()
        return d, torch.as_strided(d, self.shape, self.strides)


@pytest.fixture(scope="module")
def clip(texture_small):
    return _clip(texture_small, W, H, N)


@pytest.fixture(scope="module")
def want(clip):
    return {mode: _streaming(clip, mode, lock_at) for mode, lock_at in MODES}


def test_run_host_leaves_the_gaps_between_library_sized_frames(clip, want):
    """frames and outputs a library frame apart (388 864 bytes: 64 bytes after each frame's 388 800 pixel bytes) with
    tight rows: the outputs are the streaming ones and every byte between and after the frames is left as it was"""
    fb = 388864
    src, dst = Strided(N, H, W, 3 * W, fb), Strided(N, H, W, 3 * W, fb)
    src.frames[...] = clip
    off = offline.OfflineStabilizer(P, F, WH, H, W, B)
    off.run_host(src.buf.ctypes.data, fb, 3 * W, N, vs.GLOBAL_SMOOTHING, 0, dst.buf.ctypes.data, fb, 3 * W)
    off.close()
    assert np.array_equal(dst.frames, want[vs.GLOBAL_SMOOTHING])
    assert dst.untouched()


def test_streaming_padded_steps(clip, want):
    """host and device calls with rows padded by an odd number of bytes; call 0 (the input frame itself) included"""
    mode, lock_at = MODES[1]
    for device in (False, True):
        src, dst = Strided(1, H, W, 3 * W + 7, H * (3 * W + 7)), Strided(1, H, W, 3 * W + 13, H * (3 * W + 13))
        st = vs.Stabilizer(P, F, WH)
        if device:
            d_src, _ = src.device()
            d_dst, _ = dst.device()
        for i in range(N):
            if i == lock_at:
                st.set_stabilization_mode(mode)
            src.frames[0] = clip[i]
            if device:
                d_src.copy_(torch.from_numpy(src.buf))
                torch.cuda.synchronize()
                st.stabilize_frame_ptr(d_src.data_ptr(), H, W, src.strides[1], d_dst.data_ptr(), dst.strides[1], device=True)
                st.synchronize()
                out = d_dst.cpu().numpy()
                got = np.lib.stride_tricks.as_strided(out, dst.shape, dst.strides)[0]
            else:
                st.stabilize_frame_ptr(src.buf.ctypes.data, H, W, src.strides[1], dst.buf.ctypes.data, dst.strides[1])
                out, got = dst.buf, dst.frames[0]
            assert np.array_equal(got, want[mode][i]), (device, i)
            assert dst.untouched(out), (device, i)
        st.close()


@pytest.mark.parametrize("mode,lock_at", MODES)
def test_run_host_padded_steps(clip, want, mode, lock_at):
    src = Strided(N, H, W, 3 * W + 7, H * (3 * W + 7) + 5)
    dst = Strided(N, H, W, 3 * W + 13, H * (3 * W + 13) + 3)
    src.frames[...] = clip
    off = offline.OfflineStabilizer(P, F, WH, H, W, B)
    off.run_host(src.buf.ctypes.data, src.strides[0], src.strides[1], N, mode, lock_at, dst.buf.ctypes.data, dst.strides[0],
                 dst.strides[1])
    off.close()
    assert np.array_equal(dst.frames, want[mode])
    assert dst.untouched()


@pytest.mark.parametrize("mode,lock_at", MODES)
def test_offline_run_padded_steps(clip, want, mode, lock_at):
    """host source into host_out and into d_out"""
    src = Strided(N, H, W, 3 * W + 7, H * (3 * W + 7) + 5)
    src.frames[...] = clip
    off = offline.OfflineStabilizer(P, F, WH, H, W, B)
    off.comm_init(0, 1)
    dst = Strided(N, H, W, 3 * W + 13, H * (3 * W + 13) + 3)
    r = off.run(N, mode, lock_at, host_frames=src.frames, host_out=dst.frames)
    assert np.array_equal(dst.frames, want[mode])
    assert dst.untouched()
    dev = Strided(N, H, W, 3 * W + 13, H * (3 * W + 13) + 3)
    d_buf, d_frames = dev.device()
    r2 = off.run(N, mode, lock_at, host_frames=src.frames, device_out=d_frames)
    off.close()
    out = d_buf.cpu().numpy()
    assert np.array_equal(np.lib.stride_tricks.as_strided(out, dev.shape, dev.strides), want[mode])
    assert dev.untouched(out)
    assert np.array_equal(r["checksums"], r2["checksums"])


def test_packed_frames_move_in_one_copy(texture_small):
    """1280 x 720: the library's frame is exactly the packed frame (frame_bytes == rows * 3 * cols), so run_host and
    vstab_offline_run move a run of packed host frames in one copy each way"""
    w, h, wh, n = 1280, 720, 180, 14
    frames = _clip(texture_small, w, h, n)
    want = _streaming(frames, vs.ACCUMULATED_FULL_LOCK, 9, wh)
    off = offline.OfflineStabilizer(P, F, wh, h, w, 5)
    off.comm_init(0, 1)
    out = np.zeros_like(frames)
    off.run_host(frames.ctypes.data, frames.strides[0], frames.strides[1], n, vs.ACCUMULATED_FULL_LOCK, 9, out.ctypes.data,
                 out.strides[0], out.strides[1])
    assert np.array_equal(out, want)
    for mode, lock_at in [(vs.GLOBAL_SMOOTHING, 0), (vs.ACCUMULATED_FULL_LOCK, 9)]:
        out[:] = 0
        off.run(n, mode, lock_at, host_frames=frames, host_out=out)
        assert np.array_equal(out, want if mode == vs.ACCUMULATED_FULL_LOCK else _streaming(frames, mode, 0, wh)), mode
    off.close()
