"""Device time of bshot_detect_iss (ISS keypoints, src/lidar_odometry.cpp:447-461) against the CPU oracle.

Frames: the C3 frame (HDL-64E, 120 k points) and HDL-32E synthetic frames 0..4; parameters: the reference's defaults
(r_s 60 / r_nm 40 mm) and r_s 200 / r_nm 130 mm.  Per case: --warmup untimed calls, then --calls calls each bracketed by
CUDA events on the context stream (the call is synchronous: the window holds its launches and its one result copy),
median / p10 / p90; host wall time per call; the CPU restatement (tests/iss_oracle.cpp on the CPU oracle's radius search,
--threads OpenMP threads) median of three runs; the keypoint count; the number of (point, neighbour) pairs inside r_s and the fp64 operations of the scatter sums
(15 per pair: 3 differences, 6 products, 6 sums), from which the achieved fp64 rate of the whole call follows.
The device name and power limit are read in the same run.  Prints one JSON object (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
import iss_oracle  # noqa: E402
from conftest import load_bshot, load_oracle, load_synth  # noqa: E402


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


def pairs_within(xyz, r):
    from scipy.spatial import cKDTree
    return int(cKDTree(xyz.astype(np.float64)).query_ball_point(xyz.astype(np.float64), r, return_length=True).sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--threads", type=int, default=16, help="OpenMP threads of the CPU restatement")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.calls < 1:
        ap.error("--calls must be >= 1")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("iss_bench: no GPU (there is nothing to measure without one)")
    bs, oracle, synth = load_bshot(), load_oracle(), load_synth()
    frames = [("C3 hdl64e f0", synth.make_scan("hdl64e", 0))] + [(f"hdl32e f{k}", synth.make_scan("hdl32e", k)) for k in range(5)]
    radii = [(60.0, 40.0), (200.0, 130.0)]
    res = {"gpu": gpu_info(), "calls": args.calls, "warmup": args.warmup, "oracle_threads": args.threads, "cases": []}
    with bs.Context(0, 131072, 1024, 1024) as ctx:
        st = torch.cuda.ExternalStream(ctx.stream)
        for name, xyz in frames:
            ctx.set_cloud(xyz)
            oc = oracle.Cloud(xyz)
            for rs, rn in radii:
                p = bs.iss_default_params(salient_radius=rs, non_max_radius=rn)
                for _ in range(args.warmup):
                    g = ctx.detect_iss(p)
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.calls)]
                t0 = time.perf_counter()
                for e0, e1 in ev:
                    e0.record(st)
                    g = ctx.detect_iss(p)
                    e1.record(st)
                wall = (time.perf_counter() - t0) / args.calls
                torch.cuda.synchronize()
                ms = np.array([e0.elapsed_time(e1) for e0, e1 in ev])
                cpu = []
                for _ in range(3):
                    c0 = time.perf_counter()
                    ko = iss_oracle.iss(oc, rs, rn, threads=args.threads)
                    cpu.append(time.perf_counter() - c0)
                pairs = pairs_within(xyz, rs)
                med = float(np.median(ms))
                res["cases"].append({
                    "frame": name, "points": int(len(xyz)), "salient_radius": rs, "non_max_radius": rn,
                    "keypoints": int(len(g["idx"])), "oracle_keypoints": int(len(ko)),
                    "device_ms_median": med, "device_ms_p10": float(np.percentile(ms, 10)), "device_ms_p90": float(np.percentile(ms, 90)),
                    "host_ms_per_call": wall * 1e3, "oracle_ms_median": float(np.median(cpu)) * 1e3,
                    "speedup_vs_oracle": float(np.median(cpu)) * 1e3 / med,
                    "pairs_within_rs": pairs, "fp64_gflops_achieved": 15.0 * pairs / (med * 1e-3) / 1e9})
                print(json.dumps(res["cases"][-1]), flush=True)
    hdl32 = [c["keypoints"] for c in res["cases"] if c["frame"].startswith("hdl32e") and c["salient_radius"] == 60.0]
    res["hdl32e_iss_keypoints_per_frame_defaults"] = hdl32
    out = json.dumps(res)
    print(out)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(out + "\n")


if __name__ == "__main__":
    main()
