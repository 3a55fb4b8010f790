"""bshot_optimize_trajectory on synthetic chains of 10^3, 10^4 and 10^5 nodes with 10 and 100 loop edges (tests/test_pose_graph.py's
generator: a random walk, a drifted copy of it as the trajectory, loop edges measured from the truth with noise).

Per case: median / p90 host wall clock around the synchronous call (--warmup calls excluded), the LM iterations, the CG
iterations per LM solve against the 12 L + 1 bound, status, cost before and after.  Re-anchoring is timed by
reanchor_bench.py.  The device name and power limit are read in the same run.  Prints one JSON object (and writes it to --out)."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
from conftest import load_bshot  # noqa: E402
from relocalize_bench import gpu_info  # noqa: E402
from test_pose_graph import graph_context, synthetic  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", default="1000,10000,100000")
    ap.add_argument("--loops", default="10,100")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    bs = load_bshot()
    out = {"gpu": gpu_info(), "params": "graph_params_default()", "cases": []}
    for n in [int(v) for v in args.nodes.split(",")]:
        for L in [int(v) for v in args.loops.split(",")]:
            truth, drift, loops = synthetic(n, L, seed=n + L)
            with graph_context(bs, drift) as ctx:
                wall, r = [], None
                for i in range(args.warmup + args.reps):
                    t0 = time.perf_counter()
                    r = ctx.optimize_trajectory(loops)
                    t1 = time.perf_counter()
                    if i >= args.warmup:
                        wall.append((t1 - t0) * 1e3)
            err0 = float(np.abs(drift[:, :3, 3] - truth[:, :3, 3]).max())
            err1 = float(np.abs(r["poses"][:, :3, 3] - truth[:, :3, 3]).max())
            case = {"nodes": n, "loops": L, "wall_ms": {"median": float(np.median(wall)), "p90": float(np.percentile(wall, 90)), "n": len(wall)},
                    "iterations": r["iterations"], "cg_iterations": r["cg_iterations"],
                    "cg_per_solve": r["cg_iterations"] / max(r["iterations"], 1), "cg_bound_per_solve": 12 * L + 1, "status": r["status"],
                    "cost_initial": r["cost_initial"], "cost_final": r["cost_final"], "max_translation_error_mm": [err0, err1]}
            print(json.dumps(case), flush=True)
            out["cases"].append(case)
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
