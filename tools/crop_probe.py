"""Cost of auto-crop (vstab_set_crop / vstab_offline_set_crop) on one GPU: the same workloads with the crop off and on,
alternated in one process and repeated, median of each.

  * streaming calls/s: 1920x1080 host (pinned) buffers, working height 360, window 60/45, GLOBAL_SMOOTHING;
  * vstab_offline_run_host frames/s: the same clip and window, chunks of 16 frames;
  * config-5 style vstab_offline_run frames/s: a 3840x2160 simulator clip, working height 360, window 60/45, chunks of 128,
    one fused GLOBAL_SMOOTHING pass (the crop widens the deferred head by R calls, which a world of one does not have).

Crop on: max_zoom 1.25, release 0.002 per call (R = 125).  The card's name and power limit are read in the same run.
Prints one JSON object; --out also writes it to a file.
    python tools/crop_probe.py --out profiles/crop_n1.json
"""
import argparse
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

PAST, FUTURE, WH = 60, 45, 360
CROP = (1.25, 0.002)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, plim, clk = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:
        return {"error": str(e)[:200]}


def device_clip(torch, w, h, n):
    from vstab_b200 import offline, synth
    tex = torch.from_numpy(synth.make_texture(2048)).cuda()
    poses = synth.camera_path(n)
    frames = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda")
    offline.render_frames(tex, poses, h, w, synth.focal_for_width(w), frames)
    return frames, tex


def streaming(vs, host, calls, warmup, crop):
    n, h, w = host.shape[0], host.shape[1], host.shape[2]
    out = np.empty((h, w, 3), np.uint8)
    st = vs.Stabilizer(PAST, FUTURE, WH)
    if crop:
        st.set_crop(*CROP)
    for i in range(warmup):
        st.stabilize_frame(host[i % n], out)
    t0 = time.perf_counter()
    for i in range(calls):
        st.stabilize_frame(host[(warmup + i) % n], out)
    dt = time.perf_counter() - t0
    st.close()
    return calls / dt


def run_host(vs, host, out, crop):
    from vstab_b200 import offline
    n, h, w = host.shape[0], host.shape[1], host.shape[2]
    off = offline.OfflineStabilizer(PAST, FUTURE, WH, h, w, 16)
    if crop:
        off.set_crop(*CROP)
    args = (host.ctypes.data, host.strides[0], host.strides[1], n, vs.GLOBAL_SMOOTHING, 0, out.ctypes.data, out.strides[0],
            out.strides[1])
    off.run_host(*args)                                            # warm-up: chunk ring, output chunks, streams
    t0 = time.perf_counter()
    off.run_host(*args)
    dt = time.perf_counter() - t0
    off.close()
    return n / dt


def c5(vs, torch, tex, n, crop):
    from vstab_b200 import offline, synth
    off = offline.OfflineStabilizer(PAST, FUTURE, WH, 2160, 3840, 128)
    if crop:
        off.set_crop(*CROP)
    off.comm_init(0, 1)
    poses = synth.camera_path(n)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = off.run(n, vs.GLOBAL_SMOOTHING, 0, texture=tex, poses=poses, focal=synth.focal_for_width(3840))
    dt = time.perf_counter() - t0
    off.close()
    return n / (r["total_ms"] * 1e-3), n / dt, r["checksums"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--calls", type=int, default=600)
    ap.add_argument("--host-frames", type=int, default=512)
    ap.add_argument("--c5-frames", type=int, default=50000)
    ap.add_argument("--out")
    a = ap.parse_args()
    import torch
    import vstab_b200 as vs
    res = {"card": card(), "crop": {"max_zoom": CROP[0], "release": CROP[1]}, "window": [PAST, FUTURE], "working_height": WH}
    frames, tex = device_clip(torch, 1920, 1080, a.host_frames)
    host = torch.empty(tuple(frames.shape), dtype=torch.uint8, pin_memory=True)
    host.copy_(frames)
    host = host.numpy()
    out = torch.empty(tuple(frames.shape), dtype=torch.uint8, pin_memory=True).numpy()
    del frames
    figs = {"streaming_1080p_calls_per_s": {False: [], True: []}, "run_host_1080p_frames_per_s": {False: [], True: []},
            "c5_4k_frames_per_s": {False: [], True: []}, "c5_4k_wall_frames_per_s": {False: [], True: []}}
    for rep in range(a.reps):
        for crop in ((False, True) if rep % 2 == 0 else (True, False)):
            figs["streaming_1080p_calls_per_s"][crop].append(streaming(vs, host, a.calls, 150, crop))
            figs["run_host_1080p_frames_per_s"][crop].append(run_host(vs, host, out, crop))
            dev, wall, _ = c5(vs, torch, tex, a.c5_frames, crop)
            figs["c5_4k_frames_per_s"][crop].append(dev)
            figs["c5_4k_wall_frames_per_s"][crop].append(wall)
    for k, v in figs.items():
        off, on = statistics.median(v[False]), statistics.median(v[True])
        res[k] = {"off": off, "on": on, "change_pct": 100.0 * (on - off) / off, "off_all": v[False], "on_all": v[True]}
    res["c5_frames"] = a.c5_frames
    res["streaming_calls"], res["run_host_frames"] = a.calls, a.host_frames
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
