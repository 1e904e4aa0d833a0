"""torchrun-launched check that the N-rank sharded job (vstab_offline_run: NCCL all-gather / broadcast inside the
library) produces, call by call, the same output checksums and the same transforms as a world of one.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29511 \
      tools/verify_sharded.py [--frames 384] [--modes smooth,lock,orb,sift] [--crop MAX_ZOOM[,RELEASE]]

Every rank runs its shard of the clip (device simulator source); rank 0 additionally runs the whole clip alone on its
GPU and compares.  --crop runs both with auto-crop (vstab_offline_set_crop).  Prints one JSON line per mode on rank 0;
exit code 1 on any mismatch."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "video-stabilization_b200", "python"))

MODES = {"smooth": ("GLOBAL_SMOOTHING", 1280, 720, 360, None), "lock": ("ACCUMULATED_FULL_LOCK", 1920, 1080, 360, 46),
         "orb": ("ORB_FULL_LOCK", 1920, 1080, 1080, 46), "sift": ("SIFT_FULL_LOCK", 1920, 1080, 1080, 46)}


def main():
    import torch
    import torch.distributed as dist
    import vstab_b200 as vs
    from vstab_b200 import offline, synth
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=384)
    ap.add_argument("--modes", default="smooth,lock,orb")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--crop", help="MAX_ZOOM[,RELEASE]: auto-crop on every instance (release default: vs.CROP_RELEASE)")
    a = ap.parse_args()
    crop = [float(x) for x in a.crop.split(",")] if a.crop else None
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    tex = torch.from_numpy(synth.make_texture(2048)).cuda()
    n = a.frames
    bad = 0
    for name in a.modes.split(","):
        mname, W, H, wh, lock_at = MODES[name]
        mode = getattr(vs, mname)
        poses = synth.camera_path(n, drift=0.0 if lock_at else 0.0015)
        off = offline.OfflineStabilizer(60, 45, wh, H, W, a.batch, device=local)
        if crop:
            off.set_crop(*crop)
        off.comm_init(rank, world)
        r = off.run(n, mode, lock_at or 0, texture=tex, poses=poses, focal=synth.focal_for_width(W), want_T=True)
        off.close()
        mine = (r["call_first"], r["call_last"], r["checksums"].tolist(), r["total_ms"])
        parts = [None] * world
        if world > 1:
            dist.all_gather_object(parts, mine)
        else:
            parts = [mine]
        if rank == 0:
            solo = offline.OfflineStabilizer(60, 45, wh, H, W, a.batch, device=local)
            if crop:
                solo.set_crop(*crop)
            solo.comm_init(0, 1)
            s = solo.run(n, mode, lock_at or 0, texture=tex, poses=poses, focal=synth.focal_for_width(W), want_T=True)
            solo.close()
            got = np.zeros(n, np.uint64)
            seen = np.zeros(n, bool)
            for c0, c1, cs, _ in parts:
                got[c0:c1] = np.array(cs, np.uint64)
                seen[c0:c1] = True
            ok_cs = bool(seen.all() and np.array_equal(got, s["checksums"]))
            ok_T = bool(np.array_equal(r["T"], s["T"]))
            bad += int(not (ok_cs and ok_T))
            print(json.dumps({"mode": mname, "world": world, "frames": n, "size": [W, H], "working_height": wh, "crop": crop,
                              "checksums_equal_world1": ok_cs, "transforms_bit_equal_world1": ok_T,
                              "calls_mismatching": int((got != s["checksums"]).sum()),
                              "ms_max_over_ranks": max(p[3] for p in parts), "ms_world1": s["total_ms"]}), flush=True)
    if world > 1:
        flag = torch.tensor([bad], device="cuda")
        dist.broadcast(flag, 0)
        bad = int(flag.item())
        dist.destroy_process_group()
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
