"""Device time of bshot_voxel_grid (pcl::VoxelGrid, bshot::calculate_voxel_grid_keypoints) against the CPU reference.

Frame: the C3 frame (HDL-64E, 120 k points); leaves 100, 500, 1000 and 3000 mm.  Per leaf: --warmup untimed calls, then
--calls calls each bracketed by CUDA events on the context stream (the call is synchronous: the window holds the
host-to-device copy of the cloud, the launches and the one result copy), median / p10 / p90; host wall time per call;
the CPU reference (tests/voxel_grid_oracle.cpp, one thread) median of --cpu-runs runs; the voxel count; the bytes the
call cannot avoid moving (cloud in, records out).  The device name and power limit are read in the same run.
Prints one JSON object (and writes it to --out)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
import voxel_grid_oracle  # noqa: E402
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--cpu-runs", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.calls < 1 or args.cpu_runs < 1:
        ap.error("--calls and --cpu-runs must be >= 1")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("voxel_grid_bench: no GPU (there is nothing to measure without one)")
    bs, synth = load_bshot(), load_synth()
    L = bs.lib()
    xyz = synth.make_scan("hdl64e", 0)
    n = len(xyz)
    out = np.empty((n, 3), np.float32)
    cnt = C.c_size_t()
    res = {"gpu": gpu_info(), "frame": "C3 hdl64e f0", "points": n, "calls": args.calls, "warmup": args.warmup, "cases": []}
    with bs.Context(0, 131072, 1024, 1024) as ctx:
        st = torch.cuda.ExternalStream(ctx.stream)

        def call(leaf):
            bs._chk(L.bshot_voxel_grid(ctx.h, bs._p(xyz), n, 12, leaf, leaf, leaf, bs._p(out), n, C.byref(cnt)))

        for leaf in (100.0, 500.0, 1000.0, 3000.0):
            for _ in range(args.warmup):
                call(leaf)
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.calls)]
            t0 = time.perf_counter()
            for e0, e1 in ev:
                e0.record(st)
                call(leaf)
                e1.record(st)
            wall = (time.perf_counter() - t0) / args.calls
            torch.cuda.synchronize()
            ms = np.array([e0.elapsed_time(e1) for e0, e1 in ev])
            m = cnt.value
            same = bool(np.array_equal(out[:m].view(np.uint32), voxel_grid_oracle.voxel_grid(xyz, leaf).view(np.uint32)))
            cpu = []
            for _ in range(args.cpu_runs):
                c0 = time.perf_counter()
                voxel_grid_oracle.voxel_grid(xyz, leaf)
                cpu.append(time.perf_counter() - c0)
            med = float(np.median(ms))
            res["cases"].append({
                "leaf_mm": leaf, "voxels": int(m), "matches_cpu_reference": same,
                "device_ms_median": med, "device_ms_p10": float(np.percentile(ms, 10)), "device_ms_p90": float(np.percentile(ms, 90)),
                "host_ms_per_call": wall * 1e3, "cpu_reference_ms_median": float(np.median(cpu)) * 1e3,
                "speedup_vs_cpu_reference": float(np.median(cpu)) * 1e3 / med,
                "bytes_in_out": 12 * n + 12 * n + 16})
            print(json.dumps(res["cases"][-1]), flush=True)
    s = json.dumps(res)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
