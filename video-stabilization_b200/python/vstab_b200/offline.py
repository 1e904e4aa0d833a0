"""Offline (frame-sharded) stabilization over torch device tensors.

BASELINE.json north_star: "the frame sequence is sharded across the 8 B200s of one box by
contiguous frame ranges with halo frames.  Each GPU estimates its frame-pair transforms, a
single small NCCL all-gather over NVLink exchanges the per-frame homographies for the global
prefix accumulation and window smoothing, and each GPU then warps its own frames."

Frame pairs are independent units (corners are re-detected every frame and tracked one step,
/root/reference/src/stabilizer.cpp:1187,1318), so there is no data-path collective besides
that one all-gather of 72 bytes per frame.  The index algebra (which call presents which
frame, which transforms a call needs) is SURVEY.md Appendix C; `tests/test_sharding_gloo.py`
checks it on CPU with world_size 2 and the oracle as estimator.

torch is plumbing here (device memory, streams, torch.distributed); all pixel work happens
in libvstab.so.
"""
from __future__ import annotations

import ctypes as C

from . import (ACCUMULATED_FULL_LOCK, CROP_RELEASE, GLOBAL_SMOOTHING, SRC_DEVICE, SRC_HOST, SRC_SIMULATOR, NcclId, OfflineCfg, OfflineReport,  # noqa: F401
               ShardPlan, YuvLayout, _vp, load_library, yuv_layout_packed)
from . import _check as _check_any


def _check(st, handle=None):
    _check_any(st, handle, offline=True)        # messages of offline instances come from vstab_offline_last_error


# ----------------------------------------------------------------------------------------------
# pure index algebra (no torch, no GPU): testable on CPU
# ----------------------------------------------------------------------------------------------
def plan_shards(n_total: int, world: int):
    """Contiguous, balanced frame ranges [first, last) per rank (first ranks get the remainder)."""
    base, rem = divmod(n_total, world)
    out, first = [], 0
    for r in range(world):
        n = base + (1 if r < rem else 0)
        out.append((first, first + n))
        first += n
    return out


def calls_of_shard(first: int, last: int, n_total: int, future: int):
    """Call indices [c0, c1) whose presentation frame p(c) = max(0, c - future) lies in
    [first, last).  The owner of frame 0 also produces the `future` warm-up calls; the last
    `future` frames of a clip are never presented (SURVEY Appendix B.5)."""
    if last <= first:
        return (0, 0)
    c0 = 0 if first == 0 else first + future
    c1 = min(last + future, n_total)
    return (c0, max(c0, c1))


def padded_shard_len(n_total: int, world: int) -> int:
    return -(-n_total // world)


# ----------------------------------------------------------------------------------------------
# device runner
# ----------------------------------------------------------------------------------------------
class OfflineStabilizer:
    """One rank's share of an offline clip.  Tensors are CUDA tensors of this rank's device:
    frames uint8 [n, rows, cols, 3] (contiguous), transforms float64 [n, 9], sums int64 [n, 3]."""

    def __init__(self, past_frames: int, future_frames: int, working_height: int, rows: int, cols: int,
                 max_batch: int, device: int = 0):
        import torch
        self._torch = torch
        self._lib = load_library()
        self._h = _vp()
        self.P, self.F, self.rows, self.cols, self.max_batch, self.device = past_frames, future_frames, rows, cols, max_batch, device
        _check(self._lib.vstab_offline_create(past_frames, future_frames, working_height, rows, cols, max_batch,
                                              device, C.byref(self._h)))
        self.stream = torch.cuda.ExternalStream(int(self._lib.vstab_offline_stream(self._h)), device=device)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.vstab_offline_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _frames_ok(self, t):
        assert t.is_cuda and t.dtype == self._torch.uint8 and t.dim() == 4 and t.shape[1:] == (self.rows, self.cols, 3)
        assert t.stride(3) == 1 and t.stride(2) == 3

    def _yuv_frames_ok(self, t):
        """packed 4:2:0 frames [n, rows * 3 // 2, cols] (the frame stride may be larger than a frame)"""
        assert t.dtype == self._torch.uint8 and t.dim() == 3 and tuple(t.shape[1:]) == (self.rows * 3 // 2, self.cols)
        assert t.stride(2) == 1 and t.stride(1) == self.cols

    def set_yuv(self, in_fmt=None, out_fmt=None):
        """NV12 / I420 frames for run_host and run (vstab_offline_set_yuv): PIX_NV12 / PIX_I420 for packed frames
        [n, rows * 3 // 2, cols], a YuvLayout for any other layout, None for BGR (the default).  The clip is processed as
        BGR: checksums are those of the BGR outputs."""
        def lay(f):
            return None if f is None else f if isinstance(f, YuvLayout) else yuv_layout_packed(f, self.rows, self.cols)[0]
        self._yuv = (lay(in_fmt), lay(out_fmt))
        _check(self._lib.vstab_offline_set_yuv(self._h, *(C.byref(x) if x is not None else None for x in self._yuv)), self._h)

    def set_crop(self, max_zoom: float, release: float = CROP_RELEASE):
        """Auto-crop for render, run_host and run (vstab_offline_set_crop; see Stabilizer.set_crop).  With it on, render's
        T_all must also hold the transforms of the R calls before call_first."""
        _check(self._lib.vstab_offline_set_crop(self._h, float(max_zoom), float(release)), self._h)

    def estimate(self, frames, first: int, halo, T_out, sums_out=None):
        """T_out[i] <- transform frame (first+i-1) -> (first+i); sums_out[i] <- channel byte sums."""
        self._frames_ok(frames)
        n = frames.shape[0]
        done = 0
        while done < n:
            m = min(self.max_batch, n - done)
            h = None
            if first + done > 0:
                h = frames[done - 1] if done > 0 else halo
                assert h is not None, "halo frame required for a shard that does not start at frame 0"
            _check(self._lib.vstab_offline_estimate(
                self._h, _vp(frames[done].data_ptr()), frames.stride(0), frames.stride(1), m, first + done,
                _vp(h.data_ptr()) if h is not None else None, _vp(T_out[done].data_ptr()),
                _vp(sums_out[done].data_ptr()) if sums_out is not None else None), self._h)
            done += m

    def prepare(self, T_all, mode: int, lock_call: int = 0):
        _check(self._lib.vstab_offline_prepare(self._h, _vp(T_all.data_ptr()), T_all.shape[0], mode, lock_call), self._h)

    def render(self, frames, frame_base: int, call_first: int, ncalls: int, T_all, mode: int, lock_call: int,
               sums, out):
        """out[i] <- output of stabilizeFrame call (call_first + i); frames/sums indexed by frame - frame_base."""
        self._frames_ok(frames)
        self._frames_ok(out)
        assert out.shape[0] >= ncalls
        done = 0
        while done < ncalls:
            m = min(self.max_batch, ncalls - done)
            _check(self._lib.vstab_offline_render(
                self._h, _vp(frames.data_ptr()), frames.stride(0), frames.stride(1), frame_base, m, call_first + done,
                _vp(T_all.data_ptr()), T_all.shape[0], mode, lock_call, _vp(sums.data_ptr()),
                _vp(out[done].data_ptr()), out.stride(0), out.stride(1)), self._h)
            done += m

    def run_host(self, frames_ptr: int, frame_stride: int, step: int, n_total: int, mode: int, lock_call: int,
                 out_ptr: int, out_frame_stride: int, out_step: int):
        """Whole clip through host buffers (pointers to n_total frames in / out), pipelined uploads,
        estimation, warps and downloads; returns when the output buffer is complete."""
        _check(self._lib.vstab_offline_run_host(self._h, _vp(frames_ptr), frame_stride, step, n_total, mode, lock_call,
                                                _vp(out_ptr), out_frame_stride, out_step), self._h)

    def _yuv_in(self):
        return getattr(self, "_yuv", (None, None))[0] is not None

    def _yuv_out(self):
        return getattr(self, "_yuv", (None, None))[1] is not None

    # ---- the whole sharded job in the library (vstab_offline_run: NCCL all-gather inside) ---------------------
    def comm_init(self, rank: int, world: int, group=None):
        """Join the library-side NCCL communicator of the job: rank 0 makes the id, torch.distributed (any backend)
        only carries its 128 bytes to the other ranks."""
        import torch.distributed as dist
        nid = NcclId()
        if world > 1:
            if rank == 0:
                _check(self._lib.vstab_nccl_get_unique_id(C.byref(nid)))
            # the id is 128 opaque bytes (NULs included: read the struct's memory, not the c_char array's "string" value)
            box = [C.string_at(C.addressof(nid), C.sizeof(nid)) if rank == 0 else None]
            dist.broadcast_object_list(box, src=0, group=group)
            assert len(box[0]) == C.sizeof(nid) == 128
            C.memmove(C.addressof(nid), box[0], 128)
            _check(self._lib.vstab_offline_comm_init(self._h, C.byref(nid), rank, world), self._h)
        self.rank, self.world = rank, world

    def plan(self, n_total: int):
        pl = ShardPlan()
        _check(self._lib.vstab_offline_plan(n_total, getattr(self, "world", 1), getattr(self, "rank", 0), self.F, C.byref(pl)))
        return pl.first, pl.last, pl.call_first, pl.call_last

    def run(self, n_total: int, mode: int, lock_call: int = 0, *, texture=None, poses=None, focal: float = 0.0,
            host_frames=None, host_halo=None, host_out=None, device_frames=None, device_halo=None, device_out=None,
            want_checksums: bool = True, want_T: bool = False):
        """vstab_offline_run: this rank's share of a clip of n_total frames.  Source: `texture` (uint8 CUDA tensor
        [th, tw, 3]) + `poses` (float64 [n_total, 6]) for the device simulator, or `host_frames` (uint8 numpy / pinned
        tensor [n_local, rows, cols, 3], + `host_halo` [rows, cols, 3] on ranks > 0).  Returns a dict with the report,
        `checksums` (uint64 numpy, one per call of this rank) and optionally `T` [n_total, 3, 3].
        `device_frames` / `device_halo` / `device_out`: the shard, its halo frame and the outputs as CUDA tensors
        (resident in HBM, no staging copies).  After set_yuv, frames and outputs are packed 4:2:0 [n, rows * 3 // 2, cols]."""
        import numpy as np
        cfg = OfflineCfg()
        cfg.n_total, cfg.mode, cfg.lock_call = n_total, mode, lock_call
        keep = []
        if texture is not None:
            poses = np.ascontiguousarray(poses, np.float64)
            assert poses.shape == (n_total, 6) and texture.is_cuda and texture.is_contiguous()
            cfg.source = SRC_SIMULATOR
            cfg.d_texture, cfg.tex_rows, cfg.tex_cols = texture.data_ptr(), texture.shape[0], texture.shape[1]
            cfg.poses, cfg.focal = poses.ctypes.data_as(C.POINTER(C.c_double)), float(focal)
            keep.append(poses)
        elif device_frames is not None:
            (self._yuv_frames_ok if self._yuv_in() else self._frames_ok)(device_frames)
            cfg.source = SRC_DEVICE
            cfg.host_frames, cfg.frame_stride, cfg.step = device_frames.data_ptr(), device_frames.stride(0), device_frames.stride(1)
            cfg.host_halo = device_halo.data_ptr() if device_halo is not None else None
        else:
            cfg.source = SRC_HOST
            ptr = lambda a: a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data
            strides = lambda a: (a.stride(0), a.stride(1)) if hasattr(a, "data_ptr") else (a.strides[0], a.strides[1])
            cfg.host_frames = ptr(host_frames)
            cfg.frame_stride, cfg.step = strides(host_frames)
            cfg.host_halo = ptr(host_halo) if host_halo is not None else None
        first, last, c0, c1 = self.plan(n_total)
        if host_out is not None:
            assert host_out.shape[0] >= c1 - c0
            cfg.host_out = host_out.data_ptr() if hasattr(host_out, "data_ptr") else host_out.ctypes.data
            cfg.out_frame_stride, cfg.out_step = (host_out.stride(0), host_out.stride(1)) if hasattr(host_out, "data_ptr") \
                else (host_out.strides[0], host_out.strides[1])
        if device_out is not None:
            (self._yuv_frames_ok if self._yuv_out() else self._frames_ok)(device_out)
            assert device_out.shape[0] >= c1 - c0
            cfg.d_out, cfg.out_frame_stride, cfg.out_step = device_out.data_ptr(), device_out.stride(0), device_out.stride(1)
        sums = np.zeros(max(c1 - c0, 1), np.uint64)
        if want_checksums:
            cfg.checksums = sums.ctypes.data_as(C.POINTER(C.c_uint64))
        T = np.zeros((n_total, 9)) if want_T else None
        if want_T:
            cfg.T_all = T.ctypes.data_as(C.POINTER(C.c_double))
        rep = OfflineReport()
        _check(self._lib.vstab_offline_run(self._h, C.byref(cfg), C.byref(rep)), self._h)
        out = {k: getattr(rep, k) for k, _ in OfflineReport._fields_}
        out.update(first=first, last=last, call_first=c0, call_last=c1, checksums=sums[:c1 - c0] if want_checksums else None,
                   T=T.reshape(-1, 3, 3) if want_T else None)
        return out

    # ---- ORB / SIFT registration (frame-independent units + one broadcast + one all-gather) -----------
    def capture_reference(self, frame, mode: int):
        """Reference set from the anchor frame (uint8 [rows, cols, 3] CUDA tensor); owner rank only."""
        _check(self._lib.vstab_offline_reference_capture(self._h, _vp(frame.data_ptr()), frame.stride(0), mode), self._h)

    def export_reference(self):
        """Packed reference set as a uint8 CUDA tensor (to broadcast)."""
        t = self._torch.empty(int(self._lib.vstab_offline_reference_bytes()), dtype=self._torch.uint8,
                              device=f"cuda:{self.device}")
        _check(self._lib.vstab_offline_reference_export(self._h, _vp(t.data_ptr())), self._h)
        self.synchronize()
        return t

    def import_reference(self, pack, mode: int):
        _check(self._lib.vstab_offline_reference_import(self._h, _vp(pack.data_ptr()), mode), self._h)

    def register(self, frames, reg_out):
        """reg_out[i] (float64 [n, 10]) <- {registration matrix of frames[i] [9], valid}."""
        self._frames_ok(frames)
        _check(self._lib.vstab_offline_register(self._h, _vp(frames.data_ptr()), frames.stride(0), frames.stride(1),
                                                frames.shape[0], _vp(reg_out.data_ptr())), self._h)

    def set_registrations(self, reg_all):
        self._reg_all = reg_all          # keep alive
        _check(self._lib.vstab_offline_set_registrations(self._h, _vp(reg_all.data_ptr()), reg_all.shape[0]), self._h)

    def read_h(self, ncalls: int):
        import numpy as np
        buf = np.zeros((ncalls, 9))
        n = self._lib.vstab_offline_read_h(self._h, buf.ctypes.data_as(C.POINTER(C.c_double)), ncalls)
        return buf[:n].reshape(-1, 3, 3)

    def synchronize(self):
        _check(self._lib.vstab_offline_synchronize(self._h), self._h)

    def set_timing(self, on: bool):
        self._lib.vstab_offline_set_timing(self._h, 1 if on else 0)

    def stage_times(self):
        ms = (C.c_float * 8)()
        cnt = (C.c_int * 8)()
        _check(self._lib.vstab_offline_stage_times(self._h, ms, cnt), self._h)
        names = ("ingest", "pyramid", "gftt", "lk", "fit", "smooth", "warp", "acc_scan")
        return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(names)}


def gather_transforms(T_local, n_total: int, world: int, group=None):
    """The one collective of the path: all-gather of the per-frame 3x3 transforms
    (72 B/frame) so that every rank holds T[0..n_total).  T_local is [padded_len, 9]."""
    import torch
    import torch.distributed as dist
    if world == 1:
        return T_local[:n_total]
    pad = T_local.shape[0]
    gathered = torch.empty((world * pad, 9), dtype=T_local.dtype, device=T_local.device)
    dist.all_gather_into_tensor(gathered, T_local.contiguous(), group=group)
    shards = plan_shards(n_total, world)
    parts = [gathered[r * pad: r * pad + (l - f)] for r, (f, l) in enumerate(shards)]
    return torch.cat(parts, dim=0)


def stabilize_clip_sharded(frames_local, halo, n_total: int, rank: int, world: int, past: int, future: int,
                           estimate_fn, render_fn, gather_fn, mode: int = GLOBAL_SMOOTHING, lock_call: int = 0):
    """Backend-agnostic driver (the GPU runner and the CPU gloo test share it).

    estimate_fn(frames_local, first, halo) -> (T_local [n,9], sums_local [n,3])
    gather_fn(T_local_padded)              -> T_all [n_total, 9]
    render_fn(frames_local, frame_base, call_first, ncalls, T_all, sums_local) -> outputs
    Returns (call_first, outputs) for this rank's calls."""
    first, last = plan_shards(n_total, world)[rank]
    T_local, sums_local = estimate_fn(frames_local, first, halo)
    T_all = gather_fn(T_local)
    c0, c1 = calls_of_shard(first, last, n_total, future)
    outs = render_fn(frames_local, first, c0, c1 - c0, T_all, sums_local)
    return c0, outs


def render_frames(texture, poses, rows: int, cols: int, focal: float, out, device: int = 0):
    """CameraEngine::renderFrame for a batch of poses on the device (K13;
    /root/reference/src/camera_engine.cpp:158-172).  `texture` uint8 [th, tw, 3] and `out`
    uint8 [n, rows, cols, 3] are CUDA tensors; `poses` is a host float64 array [n, 6] of
    (x, y, z, pan, tilt, roll).  Synchronous."""
    import numpy as np
    poses = np.ascontiguousarray(poses, np.float64)
    n = poses.shape[0]
    assert out.is_cuda and out.shape[0] >= n and tuple(out.shape[1:]) == (rows, cols, 3)
    assert texture.is_cuda and texture.is_contiguous()
    lib = load_library()
    _check(lib.vstab_render_frames(device, _vp(texture.data_ptr()), texture.shape[0], texture.shape[1],
                                   poses.ctypes.data_as(C.POINTER(C.c_double)), n, rows, cols, float(focal),
                                   _vp(out.data_ptr()), out.stride(0), out.stride(1)))
