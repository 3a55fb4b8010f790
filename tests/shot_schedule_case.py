"""One schedule variant of tests/test_shot_edges.py, run as a child process: the SHOT knobs (BSHOT_SHOT_LPT,
BSHOT_SHOT_THREADS) are read into function-local statics and the grid knobs (BSHOT_YZ_MUL, BSHOT_MAX_CELLS_LOG2) at
context creation, so each setting needs a fresh process.  Writes the descriptors of fixed inputs to argv[1] (.npz)."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from conftest import load_bshot, load_synth  # noqa: E402

bshot, synth = load_bshot(), load_synth()
R = 3000.0
out = {}
with bshot.Context(0, max_points=131072, max_keypoints=20000, max_targets=20000) as ctx:
    for name, sensor, top_k in (("d64", "hdl64e", 2048), ("big", "hdl64e", 20000), ("d32", "hdl32e", 600)):
        scan = synth.make_scan(sensor, 0)
        ctx.set_cloud(scan)
        idx, _, xyz = ctx.detect_keypoints(R, 300, bshot.SR_CV, top_k)
        normals = ctx.compute_normals(bshot.NORMALS_FULL, 1000.0, 60)
        g = ctx.compute_shot(R, want_shot=True)                 # detector keypoints (LPT order when K >= 512)
        for k in ("bits", "shot", "rf", "nn"):
            out[f"{name}_det_{k}"] = g[k]
        out[f"{name}_det_sum"] = np.int64(g["sum_neighbours"])
        out[f"{name}_bin"] = ctx.binarize(g["shot"])
        ctx.set_keypoints(xyz)                                 # the same keypoints and normals, index order
        ctx.set_normals(normals)
        g = ctx.compute_shot(R, want_shot=True)
        for k in ("bits", "shot", "rf", "nn"):
            out[f"{name}_set_{k}"] = g[k]
        out[f"{name}_set_sum"] = np.int64(g["sum_neighbours"])
        out[f"{name}_idx"] = idx
        out[f"{name}_normals"] = normals
np.savez(sys.argv[1], **out)
print("schedule case ok")
