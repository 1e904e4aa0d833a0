#!/usr/bin/env python
"""bench.py -- stabilized frames/s of the LK + warp hot path (BASELINE.json configs[1]).

Workload ("c2_lk_full_lock_1080p"): synthetic 1920x1080 simulator clip (seeded texture +
scripted camera path, SURVEY.md 8d), working height 360, window 60/45, mode switched to
ACCUMULATED_FULL_LOCK at call 46.  One *step* = one pass of the whole hot path over this
rank's shard of the clip (frames resident in HBM):

    ingest(resize+gray+channel sums) -> pyramid -> Shi-Tomasi -> pyramidal LK -> RANSAC fit
    -> [all-gather of the 3x3 transforms when N > 1] -> prefix scan / window smoothing -> warp

`value`  = frames of all ranks / device time (CUDA events on the library stream, max over ranks).
`e2e`    = the same metric through the host-buffer C ABI (pinned host frames in, stabilized host
           frames out, copies inside the timed region).
`roofline` = dominant stage against the measured HBM copy bandwidth (MEASURED_PEAKS.json).
`cpu_baseline` = the oracle (cv2 restatement of the reference, all host threads) on a bounded
           sample of the same clip, rank 0 at N = 1 only.

`--impl reference` times the reference's CPU path (the oracle; the C++ binary cannot be built
offline: no OpenCV SDK) on the same config and prints the same JSON shape.

`--dump-outputs DIR` writes the stabilized frames of the last timed step (see `dump_outputs`).  The clip is
generated from fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "video-stabilization_b200", "python")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

W, H, WH = 1920, 1080, 360
PAST, FUTURE = 60, 45            # int(2.0*fps), int(1.5*fps) at the simulator's 30 fps (main.cpp:205-206)
LOCK_CALL = 46                   # setStabilizationMode(ACCUMULATED_FULL_LOCK) issued at this call (>= FUTURE)
METRIC = "stabilized_frames_per_sec_1080p_lk_full_lock"
UNIT = "frames/s"
WORKLOAD = "c2_lk_full_lock_1080p_wh360_window60_45"
# Scripted camera path of SURVEY.md 8d (jitter sigma 0.004 world units ~ 8.6 px at 1080p, +-107 px
# sinusoid, +-3 deg roll) WITHOUT its steady x drift: a full lock on a drifting camera leaves the
# anchor frame after ~500 frames and the output (and the warp's source traffic) degenerates to the
# border colour, which would flatter the warp stage.  Both arms use this same path.
PATH_DRIFT = 0.0


def shared_config():
    """The part of `config` both arms (ours / --impl reference) print identically."""
    return {"workload": WORKLOAD, "resolution": [W, H], "working_height": WH, "past": PAST, "future": FUTURE,
            "mode": "ACCUMULATED_FULL_LOCK", "lock_call": LOCK_CALL,
            "camera_path": "survey 8d jitter+sinusoid+roll, drift 0",
            "l2_policy": "inputs_exceed_l2 (every step reads its frames from memory: ours 512 x 6.2 MB of frames per GPU per "
                         "step vs 126 MB of L2; reference arm 48 distinct 1080p frames = 299 MB vs the host's last-level cache)"}


def pin_to_gpu_numa_node(torch, local):
    """Bind this process (and therefore its pinned allocations, first touch) to the CPU cores / NUMA node the GPU hangs off
    (/sys/bus/pci/devices/<bdf>/local_cpulist).  Returns a description for the JSON line."""
    info = {"bound": False}
    try:
        pr = torch.cuda.get_device_properties(local)
        # torch exposes the PCI address as three integers
        bdf = f"{int(getattr(pr, 'pci_domain_id', 0)):04x}:{int(pr.pci_bus_id):02x}:{int(pr.pci_device_id):02x}.0"
        base = f"/sys/bus/pci/devices/{bdf}"
        node = int(open(base + "/numa_node").read().strip())
        cpulist = open(base + "/local_cpulist").read().strip()
        cpus = set()
        for part in cpulist.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        before = set(os.sched_getaffinity(0))
        allowed = cpus & before
        if allowed:
            os.sched_setaffinity(0, allowed)
            info = {"bound": True, "pci": bdf, "numa_node": node, "cpus": cpulist, "n_cpus": len(allowed),
                    "restore": sorted(before)}
    except Exception as e:          # no sysfs / no permission: run unbound and say so
        info["error"] = str(e)[:80]
    return info


def working_width():
    return int(W * (WH / H))


def stage_bytes_per_frame():
    """Algorithmic (minimum) HBM bytes per frame per stage -- SURVEY.md 8d / DESIGN.md."""
    B = 3 * W * H
    px = working_width() * WH
    return {
        "ingest": B + px,
        "pyramid": px * (1 + 1 / 4 + 1 / 16) + px * (1 / 4 + 1 / 16 + 1 / 64),
        "gftt": 2 * px + 1300 * 8,
        "lk": 2 * 1.328125 * px + 1300 * 17,
        "fit": 1300 * 17 + 72,
        "smooth": 105 * 72 + 72,
        "warp": 2 * B,
        "acc_scan": 2 * 72,
    }


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(stage, frames_per_launch):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture (profiles/traffic.json,
    captured at 256 frames per launch; scaled to this run's frames per launch)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        v = t.get(stage)
        return None if v is None else float(v) * frames_per_launch / float(t.get("frames_per_launch", 256))
    except Exception:
        return None


DUMP_BYTES = 64 * 10 ** 6        # --dump-outputs: all files together
DUMP_PIXELS = 4096               # pixels per call in frames_sampled.npy
DUMP_SEED = 0


def sample_pixels(h, w, n):
    """Flat indices (y * w + x) of the n pixels of frames_sampled.npy: drawn once with DUMP_SEED, sorted."""
    return np.sort(np.random.default_rng(DUMP_SEED).choice(h * w, n, replace=False))


def dump_outputs(directory, out):
    """Writes what the timed path returned in its last step, `out` = the uint8 [ncalls, H, W, 3] device tensor of
    stabilized frames, as float32 .npy files of DUMP_BYTES at most:
      frame_last.npy      [H, W, 3]              the last call's frame, complete
      frames_sampled.npy  [ncalls, n, 3]         every call's frame at the n pixels sample_pixels(H, W, n) picks,
                                                 the same pixels in every call (n = DUMP_PIXELS unless the budget is less)"""
    import torch
    ncalls, h, w, _ = out.shape
    last = out[-1].cpu().numpy().astype(np.float32)
    n = min(DUMP_PIXELS, h * w, (DUMP_BYTES - last.nbytes - 1024) // (ncalls * 3 * 4))
    idx = torch.from_numpy(sample_pixels(h, w, n)).to(out.device)
    sampled = out.reshape(ncalls, h * w, 3).index_select(1, idx).cpu().numpy().astype(np.float32)
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "frame_last.npy"), last)
    np.save(os.path.join(directory, "frames_sampled.npy"), sampled)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        try:
            rows = [l.strip().split(", ") for l in open(self.path) if l.strip()]
            rows = [r for r in rows if len(r) >= 7]
            sm = sorted(float(r[0]) for r in rows)
            if sm:
                out["sm_mhz"] = sm[len(sm) // 2]
                out["sm_max_mhz"] = float(rows[0][1])
                out["power_w_max"] = max(float(r[2]) for r in rows)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                out["reasons"] = [n for i, n in enumerate(names) if any(r[3 + i].strip() == "Active" for r in rows)]
                out["samples"] = len(rows)
            os.unlink(self.path)
        except Exception:
            pass
        return out


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle (reference restatement over cv2) -- cpu_baseline leg and --impl reference
# ------------------------------------------------------------------------------------------------
def _render_one(args):
    from oracle import camera_engine_ref as ce
    from vstab_b200 import synth
    i, n = args
    tex = synth.make_texture(2048)
    return ce.render_frame(tex, synth.camera_path(n, drift=PATH_DRIFT)[i], W, H, synth.focal_for_width(W))


def cpu_frames(n):
    """n distinct frames of the workload clip rendered on the host (numpy restatement of CameraEngine)."""
    import multiprocessing as mp
    from vstab_b200 import synth
    synth.make_texture(2048)          # populate the on-disk cache once before forking
    procs = max(1, min(os.cpu_count() or 1, n, 32))
    with mp.get_context("fork").Pool(procs) as pool:
        return pool.map(_render_one, [(i, n) for i in range(n)])


def pingpong(i, n):
    """frame index of call i when n distinct frames are played forward/backward (motion stays small)."""
    period = 2 * (n - 1)
    j = i % period
    return j if j < n else period - j


class CpuArm:
    """Streams the workload through oracle.StabilizerRef (the reference's per-frame loop over the
    same OpenCV kernels, all quirks kept incl. GFTT twice and the three full-frame clones)."""

    def __init__(self, frames, faithful_waste=True):
        import cv2
        from oracle import stabilizer_ref as sr
        cv2.setNumThreads(os.cpu_count() or 1)
        self.cores = int(cv2.getNumThreads())
        self.sr = sr
        self.frames = frames
        self.ref = sr.StabilizerRef(PAST, FUTURE, WH, faithful_waste=faithful_waste)
        self.ref.collect_taps = False
        self.i = 0

    def run(self, ncalls):
        t0 = time.perf_counter()
        for _ in range(ncalls):
            if self.i == LOCK_CALL:
                self.ref.set_stabilization_mode(self.sr.ACCUMULATED_FULL_LOCK)
            self.ref.stabilize_frame(self.frames[pingpong(self.i, len(self.frames))])
            self.i += 1
        return time.perf_counter() - t0


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    n_distinct = args.cpu_distinct_frames
    frames = cpu_frames(n_distinct)
    arm = CpuArm(frames)
    per_step = args.cpu_frames_per_step
    for _ in range(args.warmup):
        arm.run(per_step)
    t = 0.0
    for _ in range(args.steps):
        t += arm.run(per_step)
    fps = args.steps * per_step / t
    sample = (f"{per_step} stabilizeFrame calls per step over {n_distinct} distinct 1080p simulator frames played "
              f"ping-pong, oracle.StabilizerRef (cv2 {__import__('cv2').__version__}, reference control flow incl. "
              f"GFTT x2 and frame clones), continuous stream across steps")
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/f32/f64", "data": "synthetic",
        "config": shared_config(),
        "run": {"frames_per_step": per_step, "distinct_frames": n_distinct},
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": arm.cores, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "kind=port: the C++ reference needs the OpenCV C++ SDK (absent, no network); the port calls the same "
                "OpenCV kernels through cv2 at the reference's call sites (Python overhead < 4 %)",
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import vstab_b200 as vs
    from vstab_b200 import offline, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = vs.load_library()
    numa = pin_to_gpu_numa_node(torch, local)       # before any pinned allocation: first touch decides the NUMA node

    if args.workload == "c5":
        return run_c5_line(args, torch, dist, vs, rank, world, local, numa)

    n_local = args.frames_per_gpu
    n_total = n_local * world
    first, last = offline.plan_shards(n_total, world)[rank]
    pad = offline.padded_shard_len(n_total, world)
    c0, c1 = offline.calls_of_shard(first, last, n_total, FUTURE)
    ncalls = c1 - c0

    # ---- synthetic clip, rendered on the device (K13), shard [first-1, last) ------------------------
    tex = torch.from_numpy(synth.make_texture(2048)).to(dev)
    path = synth.camera_path(n_total, drift=PATH_DRIFT)
    has_halo = first > 0
    buf = torch.empty((n_local + 1, H, W, 3), dtype=torch.uint8, device=dev)
    lo = first - 1 if has_halo else first
    chunk = 64
    for s in range(lo, last, chunk):
        e = min(last, s + chunk)
        offline.render_frames(tex, path[s:e], H, W, synth.focal_for_width(W), buf[s - lo: e - lo], device=local)
    frames = buf[1:] if has_halo else buf[:n_local]
    halo = buf[0] if has_halo else None
    out = torch.empty((max(ncalls, 1), H, W, 3), dtype=torch.uint8, device=dev)

    off = offline.OfflineStabilizer(PAST, FUTURE, WH, H, W, args.batch, device=local)
    off.comm_init(rank, world)                      # library-side NCCL communicator (the id travels over torch.distributed)
    mode = vs.ACCUMULATED_FULL_LOCK
    last_run = {}

    def step():
        # the whole sharded job behind one C-ABI call: estimate -> ncclAllGather of 72 B/frame (inside the library) ->
        # prefix scan -> smooth + warp; frames and outputs resident in HBM, per-call checksums fused into the warp
        last_run.update(off.run(n_total, mode, LOCK_CALL, device_frames=frames, device_halo=halo, device_out=out,
                                want_checksums=False))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()

    # ---- timed region -----------------------------------------------------------------------------
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    off.set_timing(True)
    off.stage_times()
    launches0 = lib.vstab_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(off.stream)
    for _ in range(args.steps):
        step()
    e1.record(off.stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = lib.vstab_launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out[:ncalls])
    # one more pass outside the timed region, with the per-call checksums (the warp's checksum variant is a few % slower)
    last_run.update(off.run(n_total, mode, LOCK_CALL, device_frames=frames, device_halo=halo, device_out=out))
    stages = off.stage_times()
    off.set_timing(False)
    clocks = sampler.stop()
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = n_total * args.steps / (ms * 1e-3)

    # ---- per-stage roofline -----------------------------------------------------------------------
    peak, peak_src = measured_peak()
    bpf = stage_bytes_per_frame()
    stage_rows = {}
    tot_stage_ms = sum(v[0] for v in stages.values()) or 1.0
    for name, (sms, cnt) in stages.items():
        if cnt == 0:
            continue
        frames_done = (n_local + (1 if has_halo and name in ("pyramid",) else 0)) * args.steps
        if name in ("smooth", "warp"):
            frames_done = ncalls * args.steps
        gbs = bpf[name] * frames_done / (sms * 1e-3) / 1e9 if sms > 0 else 0.0
        stage_rows[name] = {"ms_per_step": sms / args.steps, "share": sms / tot_stage_ms, "launches": cnt,
                            "avg_launch_ms": sms / cnt, "bytes_per_frame": bpf[name], "achieved_gbs": gbs,
                            "frac": gbs / peak}
    dom = max(stage_rows, key=lambda k: stage_rows[k]["ms_per_step"])
    d = stage_rows[dom]
    bytes_per_launch = d["achieved_gbs"] * 1e9 * d["avg_launch_ms"] * 1e-3
    roofline = {"bound": "hbm", "kernel": dom, "achieved": d["achieved_gbs"], "peak": peak, "unit": "GB/s",
                "frac": d["frac"], "traffic": ncu_traffic(dom, min(args.batch, n_local)), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": bytes_per_launch, "avg_launch_ms": d["avg_launch_ms"],
                "share_of_step": d["share"]}
    # context for the reader (not part of the contract): the whole path against the same roofline, the two stages
    # that are HBM-bound by construction, and why the dominant kernel sits far below an HBM roofline
    path_bytes = sum(bpf[k] for k in ("ingest", "pyramid", "gftt", "lk", "fit", "smooth", "warp"))
    roofline["path"] = {"algorithmic_bytes_per_frame": path_bytes, "achieved": path_bytes * value / 1e9 / max(world, 1),
                        "frac": path_bytes * value / 1e9 / max(world, 1) / peak, "unit": "GB/s per GPU"}
    roofline["hbm_bound_stages"] = {k: {"achieved": stage_rows[k]["achieved_gbs"], "frac": stage_rows[k]["frac"]}
                                    for k in ("ingest", "warp") if k in stage_rows}
    # the dominant kernel against the roofline that does bound it: warp instructions per launch (committed ncu capture, scaled
    # to this run's frames per launch) / live launch time, against SMs x 4 schedulers x the SM clock sampled during the run
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        inst = float(tj["inst"][dom]) * min(args.batch, n_local) / float(tj.get("frames_per_launch", 256))
        sms_n = torch.cuda.get_device_properties(dev).multi_processor_count
        issue_peak = sms_n * 4 * float(clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0) * 1e6
        roofline["issue"] = {"warp_instructions_per_launch": inst, "achieved_ginst_s": inst / (d["avg_launch_ms"] * 1e-3) / 1e9,
                             "peak_ginst_s": issue_peak / 1e9, "frac": inst / (d["avg_launch_ms"] * 1e-3) / issue_peak,
                             "source": "profiles/traffic.json inst (ncu smsp__inst_executed.sum of the same kernel)"}
    except Exception:
        roofline["issue"] = None
    roofline["note"] = ("the dominant kernel (pyramidal LK, one warp per feature) moves 0.6 MB of algorithmic bytes per "
                        "frame and is bound by instruction issue on the integer ALU pipe (ncu: profiles/), not by HBM; "
                        "ingest and warp are the stages an HBM roofline describes")

    # ---- e2e: host-buffer C ABI (pinned host frames in, stabilized host frames out) ------------------
    e2e = None if args.no_e2e else run_e2e(args, torch, vs, lib, frames, local, world, dev, dist)

    # ---- CPU baseline (rank 0, N = 1 only) -----------------------------------------------------------
    cpu = None
    if numa.get("restore"):
        os.sched_setaffinity(0, set(numa.pop("restore")))      # the CPU legs below get every host core again
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        nd = args.cpu_distinct_frames
        host_frames = [frames[i].cpu().numpy() for i in range(nd)]     # same bytes as the numpy renderer (tests)
        arm = CpuArm(host_frames)
        arm.run(50)
        ncpu = args.cpu_sample_frames
        t = arm.run(ncpu)
        lean = CpuArm(host_frames, faithful_waste=False)
        lean.run(50)
        nlean = max(ncpu // 2, 50)
        tl = lean.run(nlean)
        cpu = {"value": ncpu / t, "unit": UNIT, "cores": arm.cores, "kind": "port",
               "sample": f"{ncpu} stabilizeFrame calls after 50 warm-up calls over the first {nd} frames of the clip "
                         f"(ping-pong), oracle.StabilizerRef over cv2 with {arm.cores} threads; host has "
                         f"{os.cpu_count()} logical cores",
               # BASELINE.md section 3: the reference minus its obvious waste, so the speed-up is not inflated by it
               "without_reference_waste": {"value": nlean / tl, "unit": UNIT,
                                           "what": "goodFeaturesToTrack once per frame instead of twice, no full-frame clones",
                                           "sample": f"{nlean} calls after 50 warm-up calls, same frames"}}

    # ---- BASELINE config 5 (4K, simulator source, sharded over the ranks): bounded probe at every N -------------
    c5 = None
    if not args.no_c5_probe:
        halo = None
        del buf, frames, out
        torch.cuda.empty_cache()
        c5 = run_c5(args, torch, dist, vs, rank, world, local, args.c5_probe_frames, args.c5_batch)

    parity = None
    if world == 1 and rank == 0 and not args.no_parity:
        parity = run_parity(args, torch, local)

    modes, modes_offline = None, None
    if world == 1 and rank == 0 and not args.no_mode_probes:
        modes = run_mode_probes(args, torch, vs, lib, local)
        modes_offline = run_4k_probe(args, torch, vs, local, peak)
        modes_offline.update(run_feature_offline_probes(args, torch, vs, local))

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8/f32/f64", "data": "synthetic",
            "config": shared_config(),
            "run": {"frames_per_gpu": n_local, "frames_total": n_total, "batch": args.batch,
                    "api": "vstab_offline_run (VSTAB_SRC_DEVICE: shard and outputs resident in HBM)",
                    "parallelism": (f"frame-sharded x{world}, one ncclAllGather of 72 B/frame inside libvstab.so"
                                    if world > 1 else "single GPU"),
                    "numa": numa,
                    "checksum_xor_of_calls_rank0": f"{int(np.bitwise_xor.reduce(last_run['checksums'])) if len(last_run.get('checksums', [])) else 0:016x}"},
            "roofline": roofline, "stages": stage_rows, "cpu_baseline": cpu, "e2e": e2e, "parity": parity,
            "gpu_launches": int(launches), "clocks": clocks, "c5_probe": c5,
            "other_modes_streaming": modes, "other_modes_offline": modes_offline,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


C5 = dict(W=3840, H=2160, WH=360, mode="GLOBAL_SMOOTHING")


def run_c5(args, torch, dist, vs, rank, world, local, n_total, batch):
    """BASELINE config 5: offline stabilization of a synthetic 4K clip of n_total frames, frame-sharded over the ranks.
    Nothing of the clip is stored: every chunk is rendered on the device by the simulator kernel (K13) and dropped once
    its calls are warped -- GLOBAL_SMOOTHING runs as ONE fused pass of vstab_offline_run over a ring of ceil((F-1)/B)+3
    chunks (estimate chunk k, warp every call whose window is complete); only the ~P+F calls whose windows reach into a
    neighbour's shard wait for the ncclAllGather of the 3x3 transforms and have their frames rendered a second time.  The
    output of every call is reduced to a 64-bit checksum inside the warp kernel.  Strong scaling: the clip is fixed."""
    from vstab_b200 import offline, synth
    w, h, wh = C5["W"], C5["H"], C5["WH"]
    dev = torch.device("cuda", local)
    tex = torch.from_numpy(synth.make_texture(2048)).to(dev)
    poses = synth.camera_path(n_total)                       # the survey's path incl. its drift (smoothing follows it)
    off = offline.OfflineStabilizer(PAST, FUTURE, wh, h, w, batch, device=local)
    off.comm_init(rank, world)
    mode = getattr(vs, C5["mode"])
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = off.run(n_total, mode, 0, texture=tex, poses=poses, focal=synth.focal_for_width(w))
    wall = time.perf_counter() - t0
    off.close()
    cs = int(np.bitwise_xor.reduce(r["checksums"])) if len(r["checksums"]) else 0
    sm = int(r["checksums"].sum(dtype=np.uint64)) if len(r["checksums"]) else 0
    t = torch.tensor([r["total_ms"], r["source_ms"], r["estimate_ms"], r["exchange_ms"], r["render_ms"], wall * 1e3],
                     dtype=torch.float64, device=dev)
    acc = torch.tensor([cs - (1 << 64) if cs >= (1 << 63) else cs, sm - (1 << 64) if sm >= (1 << 63) else sm],
                       dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        parts = [torch.zeros_like(acc) for _ in range(world)]
        dist.all_gather(parts, acc)
    else:
        parts = [acc]
    x, sacc = 0, 0
    for pt in parts:
        a, b = int(pt[0].item()) & ((1 << 64) - 1), int(pt[1].item()) & ((1 << 64) - 1)
        x ^= a
        sacc = (sacc + b) & ((1 << 64) - 1)
    ms = [float(v) for v in t.tolist()]
    B = 3 * w * h
    calls = n_total
    return {"workload": f"c5_offline_4k_wh{wh}_{C5['mode'].lower()}_{n_total}_frames", "frames_total": n_total,
            "resolution": [w, h], "working_height": wh, "window": [PAST, FUTURE], "batch": batch,
            "value": n_total / (ms[0] * 1e-3), "unit": UNIT, "scaling": "strong", "n_gpus": world,
            "ms_total_max_over_ranks": ms[0], "wall_ms_max_over_ranks": ms[5],
            "phases_ms_max_over_ranks": {"simulator_render": ms[1], "estimate": ms[2],
                                         "exchange_allgather_plus_prefix": ms[3], "smooth_warp_checksum": ms[4]},
            "phases_note": "source, estimate and warp run on three streams and overlap: the phase times are wall intervals on their own streams and add up to more than ms_total",
            "warp_hbm_gbs": 2 * B * (calls / world) / (ms[4] * 1e-3) / 1e9 if ms[4] > 0 else None,
            "checksum_xor_of_calls": f"{x:016x}", "checksum_sum_of_calls": f"{sacc:016x}",
            "resident_frames_max": ((FUTURE - 1 + batch - 1) // batch + 1) * batch + 1,
            "api": "vstab_offline_run (VSTAB_SRC_SIMULATOR; one fused estimate + warp pass; library-side ncclAllGather; checksums fused into the warp)"}


def run_c5_line(args, torch, dist, vs, rank, world, local, numa):
    """`--workload c5`: BASELINE config 5 as the line's workload.  One step = the whole clip (default 100 000 4K frames)."""
    for _ in range(args.warmup):
        run_c5(args, torch, dist, vs, rank, world, local, min(1024, args.c5_frames), args.c5_batch)
    sampler = ClockSampler(local)
    sampler.start()
    lib = vs.load_library()
    launches0 = lib.vstab_launch_count()
    runs = [run_c5(args, torch, dist, vs, rank, world, local, args.c5_frames, args.c5_batch) for _ in range(args.steps)]
    launches = lib.vstab_launch_count() - launches0
    clocks = sampler.stop()
    ms = sum(r["ms_total_max_over_ranks"] for r in runs)
    r = runs[-1]
    peak, peak_src = measured_peak()
    if rank == 0:
        line = {"metric": "stabilized_frames_per_sec_4k_offline_sharded", "value": args.c5_frames * args.steps / (ms * 1e-3),
                "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8/f32/f64", "data": "synthetic",
                "config": {"workload": r["workload"], "resolution": r["resolution"], "working_height": r["working_height"],
                           "past": PAST, "future": FUTURE, "mode": C5["mode"], "frames_total": args.c5_frames,
                           "camera_path": "survey 8d (with drift)", "batch": args.c5_batch,
                           "l2_policy": f"inputs_exceed_l2 (every chunk of {args.c5_batch} 4K frames = {args.c5_batch * 24.9e-3:.1f} GB is rendered, read and dropped)"},
                "roofline": {"bound": "hbm", "kernel": "warp", "achieved": r["warp_hbm_gbs"], "peak": peak, "unit": "GB/s",
                             "frac": (r["warp_hbm_gbs"] or 0.0) / peak, "traffic": None, "peak_source": peak_src,
                             "note": "smooth + warp + checksum phase of the job, algorithmic 2 x 3WH bytes per frame"},
                "cpu_baseline": None, "e2e": None, "gpu_launches": int(launches), "clocks": clocks, "c5": r,
                "run": {"numa": {k: v for k, v in numa.items() if k != "restore"}},
                "note": "e2e: none -- the clip (2.5 TB) exists only on the device, chunk by chunk; the output is checksummed"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_parity(args, torch, local):
    """A bounded parity run of the headline configuration against the oracle, so that the line carries what the
    north-star tolerances look like on this very build (full-length runs: tools/parity_report.py, profiles/)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import parity_report
    try:
        r = parity_report.run("c2", args.parity_frames, check_render=0)
    except Exception as e:      # the line must still be printed
        return {"error": str(e)[:200]}
    keep = ("config", "frames", "h_px", "t_px", "t_bit_equal", "lk_bit_equal", "calls", "max_lsb", "px_gt1", "frames_gt1",
            "frac_gt1", "px_differ", "px_total")
    out = {k: r[k] for k in keep}
    out["tolerances"] = {"lk_px": 0.05, "h_px": 0.1, "pixels_lsb": 1}
    out["oracle"] = "oracle.StabilizerRef (cv2 restatement of the reference), same frames"
    return out


def run_e2e(args, torch, vs, lib, frames, local, world, dev, dist):
    """Host-buffer paths through the C ABI (include/vstab.h), pinned host memory, copies inside the
    timed region:
      * headline `value`: vstab_offline_run_host -- a whole clip of host frames in, stabilized host
        frames out (the reference's --file mode), uploads / compute / downloads pipelined;
      * `streaming`: vstab_stabilize_frame -- the reference's per-frame call, synchronous per frame."""
    from vstab_b200 import offline
    nbytes = H * W * 3
    n_clip = min(args.e2e_frames_per_step, frames.shape[0])
    lib.vstab_host_alloc.restype = C.c_void_p
    hin = lib.vstab_host_alloc(n_clip * nbytes)
    hout = lib.vstab_host_alloc(n_clip * nbytes)
    if not hin or not hout:
        raise SystemExit("pinned host allocation failed")
    hin_np = np.ctypeslib.as_array((C.c_uint8 * (n_clip * nbytes)).from_address(hin)).reshape(n_clip, H, W, 3)
    hin_np[:] = frames[:n_clip].cpu().numpy()

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(dt):
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return dt

    # ---- what the host memory system gives these ranks at the same time: a plain copy of the same pinned buffers ----
    # (names the limiter of the e2e leg at N > 1: every e2e frame is read once and written once in host DRAM by the DMA engines)
    hout_np = np.ctypeslib.as_array((C.c_uint8 * (n_clip * nbytes)).from_address(hout)).reshape(n_clip, H, W, 3)
    np.copyto(hout_np, hin_np)
    sync_all()
    t0 = time.perf_counter()
    for _ in range(2):
        np.copyto(hout_np, hin_np)
    dt_copy = max_over_ranks(time.perf_counter() - t0)
    host_copy_gbs_total = world * 2 * (2 * n_clip * nbytes) / dt_copy / 1e9      # bytes read + bytes written, all ranks

    # ---- what the links give these ranks at the same time: the same pinned buffers copied host -> device and device -> host
    # on two streams, chunked like the e2e leg, no kernels.  This is the ceiling of the e2e leg on this box at this N.
    chunk = max(1, min(args.e2e_batch, n_clip))
    secs = C.c_double(0.0)

    def link_pass(passes):
        st = lib.vstab_debug_link_probe(local, C.c_void_p(hin), C.c_void_p(hout), n_clip * nbytes, chunk * nbytes, passes, C.byref(secs))
        if st != 0:
            raise SystemExit("vstab_debug_link_probe failed")
        return secs.value
    link_pass(1)
    sync_all()
    dt_link = max_over_ranks(link_pass(2))
    link_gbs_per_gpu = 2 * n_clip * nbytes / dt_link / 1e9                        # per direction, both directions busy

    # ---- whole clip, pipelined (each rank stabilizes its own clip: replicas, no collective) --------
    off = offline.OfflineStabilizer(PAST, FUTURE, WH, H, W, args.e2e_batch, device=local)
    for _ in range(2):
        off.run_host(hin, nbytes, W * 3, n_clip, vs.ACCUMULATED_FULL_LOCK, LOCK_CALL, hout, nbytes, W * 3)
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        off.run_host(hin, nbytes, W * 3, n_clip, vs.ACCUMULATED_FULL_LOCK, LOCK_CALL, hout, nbytes, W * 3)
    dt_clip = max_over_ranks(time.perf_counter() - t0)
    off.close()

    # ---- streaming, one synchronous call per frame --------------------------------------------------
    st = vs.Stabilizer(PAST, FUTURE, WH, device=local)
    per_step = args.e2e_stream_frames
    i = 0

    def run(n):
        nonlocal i
        for _ in range(n):
            if i == LOCK_CALL:
                st.set_stabilization_mode(vs.ACCUMULATED_FULL_LOCK)
            st.stabilize_frame_ptr(hin + pingpong(i, n_clip) * nbytes, H, W, W * 3, hout, W * 3)
            i += 1

    run(max(per_step, LOCK_CALL + 4))     # warm-up incl. the mode switch
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run(per_step)
    st.synchronize()
    dt_stream = max_over_ranks(time.perf_counter() - t0)
    st.close()
    lib.vstab_host_free(C.c_void_p(hin))
    lib.vstab_host_free(C.c_void_p(hout))
    per_gpu_gbs = n_clip * nbytes * args.steps / dt_clip / 1e9
    return {"value": world * n_clip * args.steps / dt_clip, "unit": UNIT,
            "h2d_bytes_per_step": n_clip * nbytes, "d2h_bytes_per_step": n_clip * nbytes,
            # every frame crosses PCIe once per direction, both directions at the same time: the leg is bound by the link
            "pcie": {"gbs_per_direction_per_gpu": per_gpu_gbs, "frac_of_gen5_x16": per_gpu_gbs / 63.0,
                     "measured_copy_only_gbs_per_direction_per_gpu": link_gbs_per_gpu,
                     "frac_of_measured": per_gpu_gbs / link_gbs_per_gpu,
                     "measured": "pinned cudaMemcpyAsync H2D || D2H of the same buffers and chunk size on two streams, no "
                                 "kernels, all ranks at the same time (max over ranks): the ceiling of this leg on this box at this N",
                     "peak": "63.0 GB/s per direction nominal (PCIe Gen5 x16); ~55 GB/s is what pinned cudaMemcpy reaches"},
            "replicas": world,
            "host_dram": {"numpy_copy_gbs_all_ranks": host_copy_gbs_total,
                          "e2e_dma_gbs_all_ranks": 2 * world * n_clip * nbytes * args.steps / dt_clip / 1e9,
                          "note": "one single-threaded numpy copy of the same pinned buffers per rank, all ranks at once (read + "
                                  "written bytes) beside the bytes the e2e leg moves through host DRAM per second"},
            "api": "vstab_offline_run_host (whole clip of pinned host frames in/out, pipelined H2D / compute / D2H)",
            "frames_per_step": n_clip, "timer": "host wall clock around the synchronous call, max over ranks",
            "streaming": {"value": world * per_step * args.steps / dt_stream, "unit": UNIT,
                          "api": "vstab_stabilize_frame (the reference's per-frame call; synchronous, pinned host buffers)",
                          "frames_per_step": per_step, "h2d_bytes_per_step": per_step * nbytes,
                          "d2h_bytes_per_step": per_step * nbytes}}


def run_mode_probes(args, torch, vs, lib, local):
    """Secondary figures (not the headline metric): streaming frames/s of the ORB and SIFT registration
    modes at BASELINE configs 3 and 4, through the host-buffer C ABI (pinned memory)."""
    from vstab_b200 import offline, synth
    out = {}
    tex = torch.from_numpy(synth.make_texture(2048)).to(f"cuda:{local}")
    for name, w, h, wh, mode, n_distinct, n_timed in (
            ("c3_orb_full_lock_1080p_wh1080", 1920, 1080, 1080, vs.ORB_FULL_LOCK, 24, 40),
            ("c4_sift_full_lock_4k_wh2160", 3840, 2160, 2160, vs.SIFT_FULL_LOCK, 12, 16)):
        nbytes = w * h * 3
        frames = torch.empty((n_distinct, h, w, 3), dtype=torch.uint8, device=f"cuda:{local}")
        offline.render_frames(tex, synth.camera_path(n_distinct, drift=PATH_DRIFT), h, w, synth.focal_for_width(w), frames,
                              device=local)
        hin = lib.vstab_host_alloc(n_distinct * nbytes)
        hout = lib.vstab_host_alloc(nbytes)
        np.ctypeslib.as_array((C.c_uint8 * (n_distinct * nbytes)).from_address(hin)).reshape(n_distinct, h, w, 3)[:] = \
            frames.cpu().numpy()
        del frames
        st = vs.Stabilizer(PAST, FUTURE, wh, device=local)
        i = 0

        def run(n):
            nonlocal i
            for _ in range(n):
                if i == 2:
                    st.set_stabilization_mode(mode)
                st.stabilize_frame_ptr(hin + pingpong(i, n_distinct) * nbytes, h, w, w * 3, hout, w * 3)
                i += 1

        run(8)
        st.synchronize()
        t0 = time.perf_counter()
        run(n_timed)
        st.synchronize()
        dt = time.perf_counter() - t0
        cnt = st.tap(vs.TAP_ORB_COUNTS)
        st.close()
        lib.vstab_host_free(C.c_void_p(hin))
        lib.vstab_host_free(C.c_void_p(hout))
        out[name] = {"value": n_timed / dt, "unit": UNIT, "api": "vstab_stabilize_frame (streaming, pinned host buffers)",
                     "calls": n_timed, "keypoints_current": int(cnt[0]), "keypoints_reference": int(cnt[1]),
                     "matches": int(cnt[2]), "inliers": int(cnt[3])}
    return out


def run_4k_probe(args, torch, vs, local, peak):
    """Secondary figure: the LK + warp path on a 3840x2160 clip at working height 360 (the per-GPU shape of BASELINE
    config 5), frames resident in HBM, same window / mode / camera path as the headline workload."""
    from vstab_b200 import offline, synth
    w, h, wh, n = 3840, 2160, 360, 96
    dev = f"cuda:{local}"
    tex = torch.from_numpy(synth.make_texture(2048)).to(dev)
    frames = torch.empty((n, h, w, 3), dtype=torch.uint8, device=dev)
    path = synth.camera_path(n, drift=PATH_DRIFT)
    for s0 in range(0, n, 16):
        offline.render_frames(tex, path[s0:s0 + 16], h, w, synth.focal_for_width(w), frames[s0:s0 + 16], device=local)
    out = torch.empty((n, h, w, 3), dtype=torch.uint8, device=dev)
    T = torch.zeros((n, 9), dtype=torch.float64, device=dev)
    sums = torch.zeros((n, 3), dtype=torch.int64, device=dev)
    off = offline.OfflineStabilizer(PAST, FUTURE, wh, h, w, n, device=local)
    mode = vs.ACCUMULATED_FULL_LOCK

    def step():
        off.estimate(frames, 0, None, T, sums)
        off.prepare(T, mode, LOCK_CALL)
        off.render(frames, 0, 0, n, T, mode, LOCK_CALL, sums, out)

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    off.set_timing(True)
    off.stage_times()
    reps = 5
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(off.stream)
    for _ in range(reps):
        step()
    e1.record(off.stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    stages = off.stage_times()
    off.set_timing(False)
    off.close()
    B = 3 * w * h
    warp_ms = stages["warp"][0] / reps
    ingest_ms = stages["ingest"][0] / reps
    return {"c5_lk_full_lock_4k_wh360": {
        "value": n / (ms * 1e-3), "unit": UNIT, "frames": n, "ms_per_step": ms,
        "api": "vstab_offline_estimate / _prepare / _render (frames resident in HBM, one launch per stage)",
        "stages_ms": {k: v[0] / reps for k, v in stages.items() if v[1]},
        "hbm_bound_stages": {
            "ingest": {"achieved": (B + 640 * 360) * n / (ingest_ms * 1e-3) / 1e9, "frac": (B + 640 * 360) * n / (ingest_ms * 1e-3) / 1e9 / peak},
            "warp": {"achieved": 2 * B * n / (warp_ms * 1e-3) / 1e9, "frac": 2 * B * n / (warp_ms * 1e-3) / 1e9 / peak}}}}


def run_feature_offline_probes(args, torch, vs, local):
    """Secondary figures: a complete offline pass in the ORB / SIFT lock modes (BASELINE configs 3 and 4) with the frames resident
    in HBM -- LK-path estimation of the window transforms, per-frame registration against the reference set (conditioning,
    detect + describe, match, RANSAC fit; frames dealt round-robin to registration lanes), carry scan + warp."""
    from vstab_b200 import offline, synth
    out = {}
    dev = f"cuda:{local}"
    tex = torch.from_numpy(synth.make_texture(2048)).to(dev)
    for name, w, h, wh, mode, n in (("c3_orb_full_lock_1080p_wh1080", 1920, 1080, 1080, vs.ORB_FULL_LOCK, 64),
                                    ("c4_sift_full_lock_4k_wh2160", 3840, 2160, 2160, vs.SIFT_FULL_LOCK, 16)):
        frames = torch.empty((n, h, w, 3), dtype=torch.uint8, device=dev)
        path = synth.camera_path(n, drift=PATH_DRIFT)
        for s0 in range(0, n, 16):
            offline.render_frames(tex, path[s0:s0 + 16], h, w, synth.focal_for_width(w), frames[s0:s0 + 16], device=local)
        res = torch.empty((n, h, w, 3), dtype=torch.uint8, device=dev)
        T = torch.zeros((n, 9), dtype=torch.float64, device=dev)
        sums = torch.zeros((n, 3), dtype=torch.int64, device=dev)
        reg = torch.zeros((n, 10), dtype=torch.float64, device=dev)
        off = offline.OfflineStabilizer(PAST, FUTURE, wh, h, w, n, device=local)
        lock_call = FUTURE + 1                       # anchor = frame 1
        off.capture_reference(frames[lock_call - FUTURE], mode)

        def step():
            off.estimate(frames, 0, None, T, sums)
            off.register(frames, reg)
            off.set_registrations(reg)
            off.prepare(T, mode, lock_call)
            off.render(frames, 0, 0, n, T, mode, lock_call, sums, res)

        for _ in range(3):                           # the third pass replays the front ends as CUDA graphs
            step()
        torch.cuda.synchronize()
        reps = 3
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(off.stream)
        for _ in range(reps):
            step()
        e1.record(off.stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        valid = int(reg[:, 9].sum().item())
        off.close()
        del frames, res
        out[name] = {"value": n / (ms * 1e-3), "unit": UNIT, "frames": n, "ms_per_step": ms, "registrations_valid": valid,
                     "api": "vstab_offline_estimate / _register / _prepare / _render (frames resident in HBM)"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames-per-gpu", type=int, default=512)
    ap.add_argument("--batch", type=int, default=256, help="frames per kernel launch (offline batch)")
    ap.add_argument("--e2e-frames-per-step", type=int, default=512, help="frames of the host clip (one step = one clip)")
    ap.add_argument("--e2e-batch", type=int, default=16, help="chunk size of the host-clip pipeline")
    ap.add_argument("--e2e-stream-frames", type=int, default=128, help="streaming calls per step")
    ap.add_argument("--cpu-distinct-frames", type=int, default=48)
    ap.add_argument("--cpu-sample-frames", type=int, default=400)
    ap.add_argument("--cpu-frames-per-step", type=int, default=100)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs only: skip the host-buffer leg")
    ap.add_argument("--no-mode-probes", action="store_true", help="skip the ORB / SIFT streaming figures")
    ap.add_argument("--workload", default="c2", choices=["c2", "c5"], help="c5: BASELINE config 5 as the line's workload")
    ap.add_argument("--c5-frames", type=int, default=100000, help="--workload c5: frames of the 4K clip (whole job)")
    ap.add_argument("--c5-probe-frames", type=int, default=2048, help="frames of the bounded config-5 probe in the default run")
    ap.add_argument("--c5-batch", type=int, default=128, help="frames per chunk of the config-5 job (ring of 4 chunks + 1 frame resident: 12.8 GB at 4K)")
    ap.add_argument("--no-c5-probe", action="store_true")
    ap.add_argument("--parity-frames", type=int, default=160, help="frames of the bounded parity run against the oracle")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the stabilized frames of the last timed step (rank 0's "
                                                          "calls) to DIR as float32 .npy files, 64 MB at most")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "c2"):
        ap.error("--dump-outputs writes the frames of the default workload's GPU path (--impl ours --workload c2)")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
