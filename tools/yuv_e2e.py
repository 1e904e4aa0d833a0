"""End-to-end frames/s of the host-buffer paths with YUV 4:2:0 frames against BGR, on one GPU.

  * vstab_offline_run_host, the C2 configuration (1080p, working height 360, window 60/45, ACCUMULATED_FULL_LOCK from
    call 46; bench.py's e2e leg): BGR -> BGR, NV12 -> NV12 and I420 -> I420 on the same clip, alternated and repeated.
    Beside each: bytes on the host link per frame and the fraction of the ceiling that vstab_debug_link_probe (pinned
    H2D || D2H copies, no kernels) measures for that byte count.
  * vstab_stabilize_frame vs vstab_stabilize_frame_yuv (NV12): synchronous per-frame calls per second.
  * --kernels (run as a separate process by the default invocation): device time of the two K15 kernels per 1080p frame
    from torch.profiler over an NV12 run_host job, as a fraction of the 6551 GB/s HBM denominator of DESIGN section 4.

The card's name and power limit are read in the same run.  Prints one JSON object; --out also writes it to a file.
    python tools/yuv_e2e.py --out yuv_e2e.json
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "video-stabilization_b200", "python")):
    if p not in sys.path:
        sys.path.insert(0, p)

W, H, WH = 1920, 1080, 360
PAST, FUTURE, LOCK_CALL = 60, 45, 46
HBM_GBS = 6551.0                 # DESIGN section 4's HBM denominator for kernel fractions
NPIX = W * H
BGR_BYTES, YUV_BYTES = NPIX * 3, NPIX * 3 // 2


def card():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, plim, clk = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:                       # the numbers below are still worth printing
        return {"error": str(e)[:200]}


def pingpong(i, n):
    period = 2 * (n - 1)
    j = i % period
    return j if j < n else period - j


def make_clip(n):
    """n rendered 1080p frames as BGR, NV12 and I420 (cv2's conversions, which K15 matches bit for bit)"""
    import cv2
    import torch
    import vstab_b200 as vs
    from vstab_b200 import offline, synth
    tex = torch.from_numpy(synth.make_texture(2048)).cuda()
    frames = torch.empty((n, H, W, 3), dtype=torch.uint8, device="cuda")
    offline.render_frames(tex, synth.camera_path(n), H, W, synth.focal_for_width(W), frames)
    bgr = frames.cpu().numpy()
    del frames
    i420 = np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420) for f in bgr])
    nv12 = i420.copy()
    q = NPIX // 4
    c = i420[:, H:].reshape(n, -1)
    nv12[:, H:] = np.stack([c[:, :q], c[:, q:]], -1).reshape(n, H // 2, W)
    return vs, bgr, {vs.PIX_NV12: nv12, vs.PIX_I420: i420}


def pinned(lib, nbytes):
    lib.vstab_host_alloc.restype = C.c_void_p
    p = lib.vstab_host_alloc(nbytes)
    if not p:
        raise SystemExit("pinned host allocation failed")
    return p, np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(p))


def e2e(args):
    vs, bgr, yuv = make_clip(args.frames)
    from vstab_b200 import offline
    lib = vs.load_library()
    n = args.frames
    hin_bgr, a = pinned(lib, n * BGR_BYTES)
    a[:] = bgr.reshape(-1)
    hins = {0: hin_bgr}
    for fmt, clip in yuv.items():
        p, a = pinned(lib, n * YUV_BYTES)
        a[:] = clip.reshape(-1)
        hins[fmt] = p
    hout, _ = pinned(lib, n * BGR_BYTES)

    # the link's ceiling for these buffers: H2D || D2H of the BGR clip in chunks of one batch, no kernels
    secs = C.c_double(0.0)
    lib.vstab_debug_link_probe(0, C.c_void_p(hin_bgr), C.c_void_p(hout), n * BGR_BYTES, args.batch * BGR_BYTES, 1, C.byref(secs))
    if lib.vstab_debug_link_probe(0, C.c_void_p(hin_bgr), C.c_void_p(hout), n * BGR_BYTES, args.batch * BGR_BYTES, 2, C.byref(secs)):
        raise SystemExit("vstab_debug_link_probe failed")
    link_gbs = 2 * n * BGR_BYTES / secs.value / 1e9              # per direction, both directions busy

    offs = {}
    for fmt in (0, vs.PIX_NV12, vs.PIX_I420):
        o = offline.OfflineStabilizer(PAST, FUTURE, WH, H, W, args.batch)
        if fmt:
            o.set_yuv(fmt, fmt)
        offs[fmt] = o
    fb = {0: BGR_BYTES, vs.PIX_NV12: YUV_BYTES, vs.PIX_I420: YUV_BYTES}

    def run(fmt):
        o = offs[fmt]
        o.run_host(hins[fmt], fb[fmt], W * 3, n, vs.ACCUMULATED_FULL_LOCK, LOCK_CALL, hout, fb[fmt], W * 3)

    for fmt in offs:                                              # warm-up: staging buffers, events, module loads
        run(fmt)
        run(fmt)
    rates = {fmt: [] for fmt in offs}
    for _ in range(args.rounds):                                  # alternated: BGR, NV12, I420, BGR, ...
        for fmt in offs:
            t0 = time.perf_counter()
            for _ in range(args.steps):
                run(fmt)
            rates[fmt].append(n * args.steps / (time.perf_counter() - t0))
    for o in offs.values():
        o.close()
    name = {0: "bgr", vs.PIX_NV12: "nv12", vs.PIX_I420: "i420"}
    run_host = {}
    for fmt, r in rates.items():
        ceiling = link_gbs * 1e9 / fb[fmt]
        run_host[name[fmt]] = {"frames_per_s_median": statistics.median(r), "frames_per_s_all": r,
                               "link_bytes_per_frame_each_way": fb[fmt], "link_ceiling_frames_per_s": ceiling,
                               "frac_of_link_ceiling": statistics.median(r) / ceiling}
    run_host["nv12_over_bgr"] = run_host["nv12"]["frames_per_s_median"] / run_host["bgr"]["frames_per_s_median"]
    run_host["i420_over_bgr"] = run_host["i420"]["frames_per_s_median"] / run_host["bgr"]["frames_per_s_median"]

    # streaming: one synchronous call per frame, BGR against NV12, alternated
    Lnv, _ = vs.yuv_layout_packed(vs.PIX_NV12, H, W)
    stream = {"bgr": [], "nv12": []}
    sts = {"bgr": vs.Stabilizer(PAST, FUTURE, WH), "nv12": vs.Stabilizer(PAST, FUTURE, WH)}
    idx = {"bgr": 0, "nv12": 0}

    def calls(kind, k):
        st = sts[kind]
        for _ in range(k):
            i = idx[kind]
            if i == LOCK_CALL:
                st.set_stabilization_mode(vs.ACCUMULATED_FULL_LOCK)
            f = pingpong(i, n)
            if kind == "bgr":
                st.stabilize_frame_ptr(hin_bgr + f * BGR_BYTES, H, W, W * 3, hout, W * 3)
            else:
                st.stabilize_frame_yuv_ptr(hins[vs.PIX_NV12] + f * YUV_BYTES, Lnv, H, W, hout, Lnv)
            idx[kind] += 1

    for kind in sts:
        calls(kind, LOCK_CALL + 16)
    for _ in range(args.rounds):
        for kind in sts:
            t0 = time.perf_counter()
            calls(kind, args.stream_calls)
            stream[kind].append(args.stream_calls / (time.perf_counter() - t0))
    for st in sts.values():
        st.close()
    for p in list(hins.values()) + [hout]:
        lib.vstab_host_free(C.c_void_p(p))
    return {"run_host": run_host,
            "link_probe_gbs_per_direction": link_gbs,
            "streaming_calls_per_s": {k: {"median": statistics.median(v), "all": v} for k, v in stream.items()},
            "streaming_nv12_over_bgr": statistics.median(stream["nv12"]) / statistics.median(stream["bgr"])}


def kernels(args):
    """device time of the K15 kernels inside an NV12 -> NV12 run_host job (batches of `batch` frames: 9.3 MB per frame
    moved, so a batch of 16 is 149 MB, more than the 126 MB L2), per frame"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    vs, bgr, yuv = make_clip(args.batch * 4)
    from vstab_b200 import offline
    lib = vs.load_library()
    n = args.batch * 4
    hin, a = pinned(lib, n * YUV_BYTES)
    a[:] = yuv[vs.PIX_NV12].reshape(-1)
    hout, _ = pinned(lib, n * YUV_BYTES)
    o = offline.OfflineStabilizer(PAST, FUTURE, WH, H, W, args.batch)
    o.set_yuv(vs.PIX_NV12, vs.PIX_NV12)
    o.run_host(hin, YUV_BYTES, 0, n, vs.GLOBAL_SMOOTHING, 0, hout, YUV_BYTES, 0)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            o.run_host(hin, YUV_BYTES, 0, n, vs.GLOBAL_SMOOTHING, 0, hout, YUV_BYTES, 0)
        torch.cuda.synchronize()
    o.close()
    lib.vstab_host_free(C.c_void_p(hin))
    lib.vstab_host_free(C.c_void_p(hout))
    out = {}
    for ev in prof.key_averages():
        for key in ("yuv420_to_bgr_kernel", "bgr_to_yuv420_kernel"):
            if key in ev.key:
                us = (getattr(ev, "device_time", None) or getattr(ev, "cuda_time", 0.0))      # average per launch, us
                per_frame_us = us / args.batch
                gbs = (BGR_BYTES + YUV_BYTES) / (per_frame_us * 1e-6) / 1e9
                out[key] = {"launches": ev.count, "us_per_launch": us, "frames_per_launch": args.batch,
                            "us_per_1080p_frame": per_frame_us, "bytes_per_frame": BGR_BYTES + YUV_BYTES,
                            "achieved_gbs": gbs, "frac_of_6551_gbs": gbs / HBM_GBS}
    if not out:
        raise SystemExit("no K15 kernel in the trace")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=512, help="frames of the host clip (bench.py's e2e clip)")
    ap.add_argument("--batch", type=int, default=16, help="run_host chunk size (bench.py's --e2e-batch)")
    ap.add_argument("--steps", type=int, default=3, help="clips per timed sample")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the formats")
    ap.add_argument("--stream-calls", type=int, default=256, help="streaming calls per timed sample")
    ap.add_argument("--kernels", action="store_true", help="only the torch.profiler kernel timing (JSON to stdout)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this script measures the B200 and has no CPU mode")
    if args.kernels:
        print(json.dumps(kernels(args)))
        return
    res = {"config": {"W": W, "H": H, "working_height": WH, "past": PAST, "future": FUTURE, "lock_call": LOCK_CALL,
                      "frames": args.frames, "batch": args.batch, "steps": args.steps, "rounds": args.rounds},
           "card": card(), "timer": "host wall clock around synchronous calls", **e2e(args)}
    # kernel times from a separate process: tracing slows the host and must not touch the e2e numbers
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--kernels", "--batch", str(args.batch)],
                       capture_output=True, text=True)
    try:
        res["kernels"] = json.loads(r.stdout.strip().splitlines()[-1])
    except Exception:
        res["kernels"] = {"error": (r.stderr or r.stdout)[-600:]}
    res["kernels_note"] = "torch.profiler CUDA activity, separate process, inside an NV12 -> NV12 run_host job"
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
