"""Relocalisation against maps of 10^4, 10^5 and 10^6 entries (bshot_relocalize_cloud).

A real map comes from 12 HDL-32E rotations run through bshot_odometry_step; it is exported and imported again together
with distractor entries (random descriptors at the realistic <= 40-bit density, in blocks 1 km and more from the route,
beyond map_range, so ICP never sees them) until the map holds the requested number of entries.  Two queries per size:
mapped rotation 6 (preprocessed on the device, ground truth (3000, 0, 0) mm, no yaw) and a scan at an unmapped pose
(synth.make_scan at (2750, 0, 0) mm in the map frame, yaw 40 degrees, cut below the preprocessor's low-point
threshold as the mapped rotations were).  Every timed call starts from the same imported
map (the import runs before it, untimed), because an accepted relocalisation updates the map.

Per size and query: median / p90 host wall clock around the synchronous call (--warmup calls excluded), accepted, the
report's counts, and the pose error against the synthetic ground truth.  Per size, in a separate torch.profiler run:
device time per call of the matching kernels and of the RANSAC kernels.  The device name and power limit are read in the
same run.  Prints one JSON object (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
from conftest import load_bshot, load_synth  # noqa: E402

MATCH_KERNELS = ("hamming", "tc2", "mutual", "gather_best", "set_rq", "colmin", "merge")


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


def rot_z(deg):
    a = np.radians(deg)
    return np.array([[np.cos(a), -np.sin(a), 0.0], [np.sin(a), np.cos(a), 0.0], [0.0, 0.0, 1.0]])


def pose_error(T, R_true, t_true):
    T = np.asarray(T, np.float64)
    dt = float(np.linalg.norm(T[:3, 3] - np.asarray(t_true, np.float64)))
    c = (np.trace(T[:3, :3] @ np.asarray(R_true, np.float64).T) - 1.0) / 2.0
    return dt, float(np.degrees(np.arccos(np.clip(c, -1.0, 1.0))))


def distractors(synth, n, seed=11):
    rng = np.random.default_rng(seed)
    xyzr = np.empty((n, 4), np.float32)
    xyzr[:, 0] = np.round(rng.uniform(1.0e6, 1.6e6, n) / 10.0) * 10.0
    xyzr[:, 1] = np.round(rng.uniform(-3.0e5, 3.0e5, n) / 10.0) * 10.0
    xyzr[:, 2] = np.round(rng.uniform(-5.0e3, 5.0e3, n) / 10.0) * 10.0
    xyzr[:, 3] = rng.uniform(0.0, 1.0, n).astype(np.float32)
    return xyzr, synth.random_descriptors(n, seed=seed, density=40)


def real_map(bs, synth, p):
    with bs.Context(0, 131072, 1024, 1 << 16) as c:
        c.gmap_create(1 << 16, 4096)
        for k in range(12):
            L = synth.make_lasers("hdl32e", k)
            c.odometry_step(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p)
        x, d = c.gmap_export()
        L = synth.make_lasers("hdl32e", 6)
        mapped_cloud = c.preprocess(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p.vert_init_rad, p.lowpt_th)
    return x, d, mapped_cloud


def run_size(bs, synth, p, x, d, queries, size, reps, warmup):
    import torch
    dx, dd = distractors(synth, size - len(x))
    xyzr, desc = np.concatenate([x, dx]), np.concatenate([d, dd])
    out = {"entries": int(len(desc)), "real_entries": int(len(x)), "queries": {}}
    with bs.Context(0, 131072, 1024, 1 << 16) as c:
        c.gmap_create(len(desc) + 65536, 16384)
        for name, (cloud, R, t) in queries.items():
            wall, rep = [], None
            for i in range(warmup + reps):
                c.odometry_reset()
                c.gmap_import(xyzr, desc)
                t0 = time.perf_counter()
                rep = c.relocalize_cloud(cloud, p)
                t1 = time.perf_counter()
                if i >= warmup:
                    wall.append((t1 - t0) * 1e3)
            dt, da = pose_error(rep["pose"], R, t)
            out["queries"][name] = {"wall_ms": {"median": float(np.median(wall)), "p90": float(np.percentile(wall, 90)), "n": len(wall)},
                                    "accepted": int(rep["accepted"]), "n_keypoints": rep["n_keypoints"], "n_pairs": rep["n_pairs"],
                                    "n_inliers": rep["n_inliers"], "ransac_iterations": rep["ransac_iterations"],
                                    "n_icp_targets": int(rep["n_icp_targets"]), "error_mm": dt, "error_deg": da}
        # device time of matching and RANSAC per call, profiler on (a run of its own)
        from torch.profiler import ProfilerActivity, profile
        cloud = queries["mapped_rotation_6"][0]
        n_calls = 5
        c.odometry_reset()
        c.gmap_import(xyzr, desc)
        c.relocalize_cloud(cloud, p)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n_calls):
                c.odometry_reset()
                c.gmap_import(xyzr, desc)
                c.relocalize_cloud(cloud, p)
        match = ransac = 0.0
        top = []
        for e in prof.key_averages():
            t_us = getattr(e, "device_time_total", 0)
            if t_us <= 0:
                continue
            key = e.key.lower()
            if "ransac" in key:
                ransac += t_us
            elif any(k in key for k in MATCH_KERNELS):
                match += t_us
            top.append((e.key[:80], t_us / 1e3 / n_calls))
        top.sort(key=lambda r: -r[1])
        out["device_ms_per_call"] = {"matching": match / 1e3 / n_calls, "ransac": ransac / 1e3 / n_calls,
                                     "top_kernels": [{"name": k, "ms": round(v, 4)} for k, v in top[:12]]}
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
    x, d, mapped_cloud = real_map(bs, synth, p)
    novel = synth.make_scan("hdl32e", 0, pos=[2750.0, 0.0, 550.0], yaw_deg=40.0)
    novel = novel[novel[:, 2] >= p.lowpt_th]   # the preprocessor's low-point cut, which the mapped rotations went through
    queries = {"mapped_rotation_6": (mapped_cloud, np.eye(3), [3000.0, 0.0, 0.0]),
               "novel_pose_yaw40": (novel, rot_z(40.0), [2750.0, 0.0, 0.0])}
    out = {"gpu": gpu_info(), "top_k": 600, "params": "odom_default_params(top_k=600), min_inliers 15", "sizes": []}
    for size in [int(s) for s in args.sizes.split(",")]:
        out["sizes"].append(run_size(bs, synth, p, x, d, queries, size, args.reps, args.warmup))
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
