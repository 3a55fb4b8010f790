"""Re-anchoring maps of 10^4, 10^5 and 10^6 entries to a corrected trajectory (bshot_gmap_reanchor).

As in relocalize_bench.py, a real map from 12 HDL-32E rotations (bshot_odometry_step) is exported and imported again
together with distractor entries (random descriptors, blocks 1 km and more from the route) up to the requested size; the
import is update 0.  Three more steps make updates 1-3.  The timed calls then alternate between two trajectories that
differ in every update (a 0.5 degree yaw and a 200 mm shift of the whole trajectory), so every call moves every entry and
rebuilds the table; a second series re-anchors with the unchanged trajectory, which moves nothing but still rebuilds.

Per size: median / p90 host wall clock around the synchronous call (--warmup calls excluded) and, in a separate
torch.profiler run, the device time per call of the kernels.  The device name and power limit are read in the same run.
Prints one JSON object (and writes it to --out)."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
from conftest import load_bshot, load_synth  # noqa: E402
from relocalize_bench import distractors, gpu_info, rot_z  # noqa: E402


def real_map(bs, synth, p):
    with bs.Context(0, 131072, 1024, 1 << 16) as c:
        c.gmap_create(1 << 16, 4096)
        for k in range(12):
            L = synth.make_lasers("hdl32e", k)
            c.odometry_step(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p)
        return c.gmap_export()


def timed(fn, reps, warmup):
    wall = []
    for i in range(warmup + reps):
        t0 = time.perf_counter()
        fn(i)
        t1 = time.perf_counter()
        if i >= warmup:
            wall.append((t1 - t0) * 1e3)
    return {"median": float(np.median(wall)), "p90": float(np.percentile(wall, 90)), "n": len(wall)}


def run_size(bs, synth, p, x, d, size, reps, warmup):
    import torch
    from torch.profiler import ProfilerActivity, profile
    dx, dd = distractors(synth, size - len(x))
    xyzr, desc = np.concatenate([x, dx]), np.concatenate([d, dd])
    with bs.Context(0, 131072, 1024, 1 << 16) as c:
        c.gmap_create(len(desc) + 65536, 16384)
        c.gmap_import(xyzr, desc)
        for k in (4, 5, 6):
            L = synth.make_lasers("hdl32e", k)
            c.odometry_step(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p)
        entries = c.gmap_size()[0]
        _, traj = c.gmap_scans()
        D = np.eye(4)
        D[:3, :3], D[:3, 3] = rot_z(0.5), [200.0, -100.0, 0.0]
        moved = (D @ traj.astype(np.float64)).astype(np.float32)
        moved[:, 3] = [0, 0, 0, 1]
        pair = (moved, traj)
        out = {"entries": int(entries), "real_entries": int(len(x)), "updates": int(len(traj))}
        out["all_moved_wall_ms"] = timed(lambda i: c.gmap_reanchor(pair[i % 2]), reps, warmup)
        c.gmap_reanchor(traj)
        out["unchanged_wall_ms"] = timed(lambda i: c.gmap_reanchor(traj), reps, warmup)
        n_calls = 6
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(n_calls):
                c.gmap_reanchor(pair[i % 2])
        total, top = 0.0, []
        for e in prof.key_averages():
            t_us = getattr(e, "device_time_total", 0)
            if t_us <= 0:
                continue
            total += t_us
            top.append((e.key[:80], t_us / 1e3 / n_calls))
        top.sort(key=lambda r: -r[1])
        out["device_ms_per_call"] = {"total": total / 1e3 / n_calls, "top": [{"name": k, "ms": round(v, 4)} for k, v in top[:10]]}
        assert c.gmap_size()[0] == entries
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="10000,100000,1000000")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    bs, synth = load_bshot(), load_synth()
    p = bs.odom_default_params(top_k=600)
    x, d = real_map(bs, synth, p)
    out = {"gpu": gpu_info(), "sizes": []}
    for size in [int(s) for s in args.sizes.split(",")]:
        out["sizes"].append(run_size(bs, synth, p, x, d, size, args.reps, args.warmup))
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
