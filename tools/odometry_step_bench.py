"""The per-scan odometry step (bshot_odometry_step, one call) against the five-call chain it replaces (bshot_extract_scan,
bshot_match_mutual / bshot_match_frame_to_map, bshot_ransac, bshot_evaluate_estimation, bshot_gmap_update_from_frame +
bshot_frame_commit), in one process on the same rotations, alternating the two arms frame by frame.

Configs: 12 HDL-32E rotations at K = 600 (bench.py's pose_loop) and --frames64 HDL-64E rotations at K = 2048.  Each arm
has its own context and map.  One full untimed pass warms both up (module load, scratch growth); then --passes timed passes,
each after a reset of both arms.  Per arm: median and p90 host wall clock per frame (first, INITIAL-status frame excluded);
for the step also the CUDA-event span on the context stream (the step ends in a device synchronise, so the span holds the
launches, the preprocessor's two count read-backs and the report copy).  Every frame's pose must be identical in both arms.
The device name and power limit are read in the same run.  Prints one JSON object (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
from conftest import load_bshot, load_synth  # noqa: E402


def gpu_info():
    import torch
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                                    text=True, timeout=30).strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except (OSError, subprocess.SubprocessError, ValueError) as e:
        info["power_limit"] = f"not read ({e.__class__.__name__})"
    return info


def chain(ctx, L, p, state):
    """the five calls of tests/test_odometry_loop.py / bench.py:bench_pose_loop"""
    f = ctx.extract_scan(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p.front, vert_init=p.vert_init_rad, lowpt_th=p.lowpt_th,
                         want_cloud=False)
    pose_ref = state["pose"]
    if state["initial"]:
        pairs, tgt = ctx.match_mutual(f["bits"], f["bits"])[0], f["kp_xyz"]
    else:
        r = ctx.match_frame_to_map(pose_ref[:3, 3], p.map_range, pose_ref[:3], target_cap=1 << 17)
        pairs, tgt = r["pairs"], r["target_xyz"]
    rs = ctx.ransac(f["kp_xyz"], tgt, pairs, p.ransac_iterations, p.inlier_threshold)
    ev = ctx.evaluate_estimation(rs["transform"], pose_ref, len(rs["pairs"]), f["kp_xyz"], tgt, run_icp=bool(p.run_icp))
    ctx.gmap_update_from_frame(ev["T_best"][:3])
    ctx.frame_commit()
    ctx.sync()
    state["pose"], state["initial"] = ev["T_best"], False
    return ev["T_best"]


def run_config(bs, rots, top_k, passes, max_points, max_kp, profile=False):
    import torch
    p = bs.odom_default_params(top_k=top_k)
    a = bs.Context(0, max_points, max_kp, 1 << 17)
    b = bs.Context(0, max_points, max_kp, 1 << 17)
    a.gmap_create(1 << 17, 4096)
    b.gmap_create(1 << 17, 4096)
    sb = torch.cuda.ExternalStream(b.stream)
    wall = {"chain": [], "step": []}
    dev = []
    for rep in range(passes + 1):   # pass 0 warms up
        a.reset(); a.gmap_reset(); b.odometry_reset()
        state = dict(pose=np.eye(4, dtype=np.float32), initial=True)
        for k, L in enumerate(rots):
            t0 = time.perf_counter()
            Ta = chain(a, L, p, state)
            t1 = time.perf_counter()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(sb)
            r = b.odometry_step(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p)
            e1.record(sb)
            t2 = time.perf_counter()
            e1.synchronize()
            assert np.array_equal(Ta.view(np.uint32), r["pose"].view(np.uint32)), (rep, k)
            if rep > 0 and k > 0:
                wall["chain"].append((t1 - t0) * 1e3)
                wall["step"].append((t2 - t1) * 1e3)
                dev.append(e0.elapsed_time(e1))
    n_map = b.gmap_size()[0]
    assert a.gmap_size()[0] == n_map
    kernels = None
    if profile:   # where the step's device time goes: per-kernel device time per step over one more pass (tracing on)
        from torch.profiler import ProfilerActivity, profile as tprofile
        b.odometry_reset()
        with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
            for L in rots:
                b.odometry_step(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p)
        rows = [(e.key, e.device_time_total / 1e3 / len(rots), e.count / len(rots)) for e in prof.key_averages()
                if getattr(e, "device_time_total", 0) > 0]
        rows.sort(key=lambda r: -r[1])
        kernels = [{"name": k[:80], "ms_per_step": round(t, 4), "launches_per_step": round(c, 2)} for k, t, c in rows[:25]]
    a.close(); b.close()

    def stats(v):
        return {"median": float(np.median(v)), "p90": float(np.percentile(v, 90)), "n": len(v)}
    return {"frames": len(rots), "top_k": top_k, "chain_wall_ms": stats(wall["chain"]), "step_wall_ms": stats(wall["step"]),
            "step_device_span_ms": stats(dev), "map_keypoints": int(n_map), "poses_identical": True,
            "last_position_mm": [float(x) for x in r["pose"][:3, 3]], "step_kernels": kernels}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--frames64", type=int, default=8)
    ap.add_argument("--out", default="")
    ap.add_argument("--profile", action="store_true", help="add the step's per-kernel device times (torch.profiler, separate pass)")
    args = ap.parse_args()
    bs, synth = load_bshot(), load_synth()
    out = {"gpu": gpu_info(), "passes": args.passes,
           "hdl32e_k600": run_config(bs, [synth.make_lasers("hdl32e", f) for f in range(12)], 600, args.passes, 131072, 1024, args.profile),
           "hdl64e_k2048": run_config(bs, [synth.make_lasers("hdl64e", f) for f in range(args.frames64)], 2048, args.passes, 1 << 18, 4096, args.profile)}
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
