"""Loop detection against maps of 10^4, 10^5 and 10^6 candidate entries (bshot_detect_loop).

A real map comes from 12 HDL-32E rotations run through bshot_odometry_step; it is exported and imported again together
with distractor entries (random descriptors at the realistic <= 40-bit density, in blocks 1 km and more from the route,
beyond map_range, so ICP never sees them) until the map holds the requested number of entries.  All of them are the
import's update 0.  One step then takes mapped rotation 6 again (a revisit; the step is update 1, INITIAL, so its pose
is the identity while the map places it at (3000, 0, 0) mm), and detect_loop with min_gap = 1 searches every imported
entry.  The detection is read only, so the timed calls repeat on the same state.

Per size: median / p90 host wall clock around the synchronous call (--warmup calls excluded), the report's counts and
T_rel's error against the 3000 mm ground truth.  In a separate torch.profiler run: device time per call of the
whole-map gather and candidate filter, the matching, RANSAC, ICP and the vote kernels.  The device name and power
limit are read in the same run.  Prints one JSON object (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
from conftest import load_bshot, load_synth  # noqa: E402

# profiler kernel name -> stage (first match wins)
STAGES = (("vote_final", ("loop_final",)), ("gather_filter", ("gm_", "rx_")), ("ransac", ("ransac",)), ("icp", ("icp",)),
          ("matching", ("hamming", "tc2", "mutual", "gather_best", "set_rq", "colmin", "merge")))


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


def pose_error(T, t_true):
    T = np.asarray(T, np.float64)
    dt = float(np.linalg.norm(T[:3, 3] - np.asarray(t_true, np.float64)))
    c = (np.trace(T[:3, :3]) - 1.0) / 2.0
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
        return c.gmap_export()


def run_size(bs, synth, p, lp, x, d, size, reps, warmup):
    import torch
    dx, dd = distractors(synth, size - len(x))
    xyzr, desc = np.concatenate([x, dx]), np.concatenate([d, dd])
    out = {"entries": int(len(desc)), "real_entries": int(len(x))}
    with bs.Context(0, 131072, 1024, 1 << 16) as c:
        c.gmap_create(len(desc) + 65536, 16384)
        c.gmap_import(xyzr, desc)
        L = synth.make_lasers("hdl32e", 6)
        c.odometry_step(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p)
        wall, rep = [], None
        for i in range(warmup + reps):
            t0 = time.perf_counter()
            rep = c.detect_loop(lp)
            t1 = time.perf_counter()
            if i >= warmup:
                wall.append((t1 - t0) * 1e3)
        dt, da = pose_error(rep["T_rel"], [3000.0, 0.0, 0.0])
        out.update({"wall_ms": {"median": float(np.median(wall)), "p90": float(np.percentile(wall, 90)), "n": len(wall)},
                    "accepted": int(rep["accepted"]), "match_scan": rep["match_scan"], "votes": rep["votes"], "n_candidates": int(rep["n_candidates"]),
                    "n_keypoints": rep["n_keypoints"], "n_pairs": rep["n_pairs"], "n_inliers": rep["n_inliers"],
                    "ransac_iterations": rep["ransac_iterations"], "n_icp_targets": int(rep["n_icp_targets"]), "T_rel_error_mm": dt,
                    "T_rel_error_deg": da})
        # device time per call by stage, profiler on (a run of its own)
        from torch.profiler import ProfilerActivity, profile
        n_calls = 5
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n_calls):
                c.detect_loop(lp)
        stages = {name: 0.0 for name, _ in STAGES}
        stages["other"] = 0.0
        top = []
        for e in prof.key_averages():
            t_us = getattr(e, "device_time_total", 0)
            if t_us <= 0:
                continue
            key = e.key.lower()
            stage = next((name for name, keys in STAGES if any(k in key for k in keys)), "other")
            stages[stage] += t_us / 1e3 / n_calls
            top.append((e.key[:80], t_us / 1e3 / n_calls))
        top.sort(key=lambda r: -r[1])
        out["device_ms_per_call"] = {k: round(v, 4) for k, v in stages.items()}
        out["top_kernels"] = [{"name": k, "ms": round(v, 4)} for k, v in top[:12]]
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
    lp = bs.loop_params_default(min_gap=1)
    x, d = real_map(bs, synth, p)
    out = {"gpu": gpu_info(), "top_k": 600, "params": "odom_default_params(top_k=600), loop_params_default(min_gap=1)", "sizes": []}
    for size in [int(s) for s in args.sizes.split(",")]:
        out["sizes"].append(run_size(bs, synth, p, lp, x, d, size, args.reps, args.warmup))
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
