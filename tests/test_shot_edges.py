"""SHOT's rare paths on the GPU against the float64 reference (tests/shot_f64.py).

Every descriptor below is judged by `shot_f64.check_shot`: per-bin bounds from the bin's vote count and the
kernel's fixed-point resolution, the support, and the B-SHOT bits near a threshold only.  Every call also checks
that the bits written by compute_shot equal the standalone binariser applied to its floats."""
import os
import subprocess
import sys

import numpy as np
import pytest

import shot_f64 as sf
from test_shot_f64 import PREF_A, PREF_B, SHELL_RADII, blob, tie_set

pytestmark = pytest.mark.gpu
f32 = np.float32
HERE = os.path.dirname(os.path.abspath(__file__))
REACHED = {}                                                  # largest |g - r| / bound per case, printed with -s


def shot_gpu(ctx, pts, kp, normals, R):
    ctx.set_cloud(pts)
    ctx.set_keypoints(kp)
    ctx.set_normals(normals)
    g = ctx.compute_shot(R, want_shot=True)
    assert np.array_equal(g["bits"], ctx.binarize(g["shot"]))   # the two binarisers agree bit for bit
    return g


def judge(case, pts, kp, normals, R, g, which):
    """check_shot on keypoints `which`; neighbour counts exact; returns the largest excess"""
    worst, nib = 0.0, 0
    for i in which:
        ref = sf.shot_f64(pts, kp[i], R, normals, g["rf"][i])
        assert g["nn"][i] == ref["n_all"], (case, i)
        c = sf.check_shot(g["shot"][i], g["bits"][i:i + 1], ref, sf.fx_bits(ref["n_all"]))
        assert c["ok"], (case, i, ref["n_all"], c["why"])
        worst, nib = max(worst, c["excess"]), nib + c["nib_diff"]
    REACHED[case] = (worst, nib)
    print(f"{case}: max |g-r|/bound {worst:.3g}, {nib} nibbles off the binarised reference")
    return worst


# ---- 1. half-radius shell -------------------------------------------------------------------------------------

@pytest.mark.parametrize("R", SHELL_RADII + [3000.0])
def test_shell_boundary(gpu_ctx, R):
    """neighbours at sqd == fl(R^2/4) and one fp32 step below / above it, each on its own axis"""
    x = f32(R / 2)
    lo, hi = np.nextafter(x, f32(0)), np.nextafter(x, f32(np.inf))
    assert float(x * x) == float(f32(float(f32(R)) ** 2 / 4))
    bg = np.array([[0.2, 0.1, 0.05], [-0.3, 0.2, -0.1], [0.1, -0.7, 0.2], [-0.2, -0.1, 0.8], [0.6, 0.5, -0.3]]) * R
    pts = np.concatenate([[[0, 0, 0], [x, 0, 0], [0, -lo, 0], [0, 0, hi], [-x, 0, 0]], bg]).astype(f32)
    rng = np.random.default_rng(1)
    normals = rng.normal(0, 1, (len(pts), 4)).astype(f32)
    normals[:, :3] /= np.linalg.norm(normals[:, :3], axis=1, keepdims=True).astype(f32)
    g = shot_gpu(gpu_ctx, pts, pts[:1], normals, R)
    ref = sf.shot_f64(pts, pts[0], R, normals, g["rf"][0])
    assert g["sum_neighbours"] == ref["n_all"] == len(pts)
    c = sf.check_shot(g["shot"][0], g["bits"], ref, sf.fx_bits(ref["n_all"]))   # bin for bin
    assert c["ok"], c["why"]


# ---- 2. float64 comparison at scale ------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def scans(synth):
    return {s: synth.make_scan(s, 0) for s in ("hdl32e", "hdl64e")}


@pytest.mark.parametrize("mode", ["full", "reference"])
@pytest.mark.parametrize("R", [700.0, 1500.0, 3000.0, 5000.0, 8000.0])
@pytest.mark.parametrize("sensor", ["hdl32e", "hdl64e"])
def test_scan_against_f64(gpu_ctx, bshot, scans, sensor, R, mode):
    """R = 8000 mm: the query rectangle holds > 1024 grid rows (the multi-pass neighbour walk)"""
    pts = scans[sensor]
    rng = np.random.default_rng(int(R) + len(pts))
    kp = pts[np.sort(rng.choice(len(pts), 256, replace=False))]
    gpu_ctx.set_cloud(pts)
    gpu_ctx.set_keypoints(kp)
    if mode == "full":
        normals = gpu_ctx.compute_normals(bshot.NORMALS_FULL, 1000.0, 60)
    else:                                                       # keypoint normals at surface indices 0..K-1, zeros after
        normals = gpu_ctx.compute_normals(bshot.NORMALS_REFERENCE, R, 300)
    g = shot_gpu(gpu_ctx, pts, kp, normals, R)
    which = rng.choice(len(kp), 12 if R >= 5000 else 24, replace=False)
    judge(f"{sensor} R={R:g} {mode}", pts, kp, normals, R, g, which)


@pytest.mark.parametrize("n, fx", [(120_000, 13), (2_000_000, 9)])
def test_dense_blob_against_f64(bshot, gpu_ctx, n, fx):
    """> 65 536 candidates per query (the batch table's binary-search tail) and the coarse fixed-point grid"""
    pts, normals = blob(n, 11, (500.0, 350.0, 150.0))
    kp = np.array([[0, 0, 0], [300, -200, 50], [-400, 100, -100], [150, 250, 120]], f32)
    if n <= gpu_ctx.max_points:
        g = shot_gpu(gpu_ctx, pts, kp, normals, 3000.0)
    else:
        with bshot.Context(0, max_points=n, max_keypoints=64, max_targets=64) as ctx:
            g = shot_gpu(ctx, pts, kp, normals, 3000.0)
    assert all(sf.fx_bits(int(m)) == fx for m in g["nn"])
    judge(f"blob {n}", pts, kp, normals, 3000.0, g, range(len(kp)))


# ---- 3. LRF exact ties ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("pref", [PREF_A, PREF_B], ids=["x_flip_z_keep", "x_keep_z_flip"])
@pytest.mark.parametrize("shell", [False, True], ids=["fast_path", "radix_select"])
def test_lrf_exact_ties(gpu_ctx, oracle, shell, pref):
    pts = tie_set(80 if shell else 6, shell, 3, pref)
    L = sf.lrf_f64(pts, pts[0], 3000.0)
    assert L["tie"] == (True, True)                             # s == 0 on both axes
    gpu_ctx.set_cloud(pts)
    gpu_ctx.set_keypoints(pts[:1])
    rf, nv = gpu_ctx.compute_lrf(3000.0)
    assert nv[0] == L["n_valid"]
    rf_o, _ = oracle.Cloud(pts).lrf(pts[:1], 3000.0)
    assert np.abs(rf[0] - L["rf"]).max() <= 1e-6 and np.abs(rf[0] - rf_o[0]).max() <= 1e-6
    rng = np.random.default_rng(2)
    normals = rng.normal(0, 1, (len(pts), 4)).astype(f32)
    normals[:, :3] /= np.linalg.norm(normals[:, :3], axis=1, keepdims=True).astype(f32)
    g = shot_gpu(gpu_ctx, pts, pts[:1], normals, 3000.0)
    # The neighbour walk lists a query's grid rows in the order the threads claim them (atomicAdd), so the fp64
    # covariance is summed in an order that can change from launch to launch.  The true off-diagonal terms of this
    # set are zero, so the rounding residue (~1e-18) is all that remains of them and survives into the fp32 frame:
    # two launches agree on the axes and their signs, not on those residues.
    assert np.abs(g["rf"][0] - rf[0]).max() <= 1e-6 and np.abs(g["rf"][0] - L["rf"]).max() <= 1e-6
    judge(f"ties {'shell' if shell else 'few'}", pts, pts[:1], normals, 3000.0, g, [0])


# ---- 4. degenerate inputs ------------------------------------------------------------------------------------------

def test_degenerate_inputs(gpu_ctx, oracle):
    R = 3000.0
    rng = np.random.default_rng(9)
    sym = tie_set(6, False, 5, PREF_A)[1:]                      # axis-aligned rf about the origin
    a, b, c = 700.0, 400.0, 150.0
    edges = [(s1 * a, s2 * a, s3 * c) for s1 in (1, -1) for s2 in (1, -1) for s3 in (1, -1)]       # x = +-y
    edges += [(0.0, s1 * b, s2 * c) for s1 in (1, -1) for s2 in (1, -1)]                            # x = 0
    edges += [(s1 * b, 0.0, s2 * c) for s1 in (1, -1) for s2 in (1, -1)]                            # y = 0
    edges += [(s1 * a, s2 * b, 0.0) for s1 in (1, -1) for s2 in (1, -1)]                            # z = 0
    far = np.array([50000.0, 0, 0])
    few4 = far + np.array([[100, 0, 0], [0, 100, 0], [0, 0, 100], [-100, 0, 0]])
    few5 = 2 * far + np.array([[100, 0, 0], [0, 60, 0], [0, 0, 30], [-90, 0, 0], [0, -50, 10]])   # distinct eigenvalues
    dup = np.array([[20000.0, 5000, 0]] * 3)                   # three cloud points equal to the keypoint
    dup_nb = dup[0] + rng.uniform(-800, 800, (12, 3))
    pts = np.concatenate([[[0, 0, 0]], sym, edges, few4, few5, dup, dup_nb]).astype(f32)
    normals = rng.normal(0, 1, (len(pts), 4)).astype(f32)
    normals[:, :3] /= np.linalg.norm(normals[:, :3], axis=1, keepdims=True).astype(f32)
    normals[len(sym) + 3, 0] = np.nan
    normals[len(sym) + 7, 2] = np.inf
    normals[-2, 1] = -np.inf
    kp = np.array([[0, 0, 0], [np.nan, 0, 0], [-90000, 0, 0], far, 2 * far, dup[0]], f32)
    gpu_ctx.set_cloud(pts)
    gpu_ctx.set_keypoints(kp)
    rf_l, nv = gpu_ctx.compute_lrf(R)
    g = shot_gpu(gpu_ctx, pts, kp, normals, R)
    oc = oracle.Cloud(pts)
    rf_o, nv_o = oc.lrf(kp, R)
    so, _, nn_o, tot_o = oc.shot(kp, normals, R)
    n_all = [sf.shot_f64(pts, q, R, normals, np.eye(3, dtype=f32).ravel())["n_all"] for q in kp]
    n_valid = [sf.lrf_f64(pts, q, R)["n_valid"] for q in kp]
    assert list(nv) == list(nv_o) == n_valid                    # compute_lrf: neighbours other than the keypoint
    assert list(g["nn"]) == list(nn_o) == n_all                 # compute_shot: every neighbour
    assert g["sum_neighbours"] == tot_o == sum(n_all)
    assert n_valid[5] == 12 and n_all[5] == 15 and n_all[3] == 4 and n_all[4] == 5 and n_all[1] == n_all[2] == 0
    nan_g, nan_o = np.isnan(g["shot"]).any(1), np.isnan(so).any(1)
    assert np.array_equal(nan_g, nan_o) and list(np.nonzero(nan_g)[0]) == [1, 2, 3]   # < 5 neighbours: NaN
    assert (g["bits"][nan_g] == np.uint64(0xFFFFFFFFFFFFFFFF))[:, :5].all()
    ok = ~nan_o
    assert np.array_equal(np.isnan(rf_l).any(1), ~ok)
    # the points with x = 0 or z = 0 make the origin's sign votes depend on rounding noise: compare the frames of the
    # other keypoints with the oracle, and the origin's only up to the signs of its axes
    assert np.abs(rf_l[[4, 5]] - rf_o[[4, 5]]).max() <= 1e-4
    assert np.abs(np.abs(g["rf"][0]) - np.eye(3, dtype=f32).ravel()).max() <= 1e-6
    judge("degenerate", pts, kp, normals, R, g, np.nonzero(ok)[0])


# ---- 5. only the schedule may differ --------------------------------------------------------------------------------

VARIANTS = {"default": {}, "lpt0": {"BSHOT_SHOT_LPT": "0"}, "threads64": {"BSHOT_SHOT_THREADS": "64"},
            "threads256": {"BSHOT_SHOT_THREADS": "256"}, "yz2": {"BSHOT_YZ_MUL": "2"}, "cells10": {"BSHOT_MAX_CELLS_LOG2": "10"}}


@pytest.fixture(scope="module")
def schedule_runs(tmp_path_factory):
    d = tmp_path_factory.mktemp("shot_schedule")
    runs = {}
    for name, env in VARIANTS.items():
        e = {k: v for k, v in os.environ.items() if k not in ("BSHOT_SHOT_LPT", "BSHOT_SHOT_THREADS", "BSHOT_YZ_MUL", "BSHOT_MAX_CELLS_LOG2")}
        e.update(env)
        out = d / f"{name}.npz"
        r = subprocess.run([sys.executable, os.path.join(HERE, "shot_schedule_case.py"), str(out)], env=e,
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and "schedule case ok" in r.stdout, (name, r.stdout[-2000:], r.stderr[-2000:])
        runs[name] = dict(np.load(out))
    return runs


def same(a, b, keys):
    return all(np.array_equal(a[k], b[k], equal_nan=np.issubdtype(a[k].dtype, np.floating)) for k in keys)


def test_detector_order_equals_index_order(schedule_runs):
    """LPT order (K = 600, 2048) and the K > 16 384 plain-order branch against the same keypoints given in index order"""
    for r in schedule_runs.values():
        for name in ("d32", "d64", "big"):
            for k in ("bits", "shot", "rf", "nn", "sum"):
                assert np.array_equal(r[f"{name}_det_{k}"], r[f"{name}_set_{k}"], equal_nan=k in ("shot", "rf")), (name, k)
            assert np.array_equal(r[f"{name}_det_bits"], r[f"{name}_bin"])
    assert len(schedule_runs["default"]["big_idx"]) > 16384 and len(schedule_runs["default"]["d64_idx"]) >= 512


def test_lpt_off_is_bit_identical(schedule_runs):
    d, v = schedule_runs["default"], schedule_runs["lpt0"]
    for name in ("d32", "d64", "big"):
        assert same(d, v, [f"{name}_det_{k}" for k in ("bits", "shot", "rf", "nn", "sum")]), name


@pytest.mark.parametrize("variant", ["threads64", "threads256", "yz2", "cells10"])
def test_summation_order_knobs(synth, schedule_runs, variant):
    """these change the order of the fp64 covariance sums: rf within 1e-6, descriptors within the float64 bound"""
    d, v = schedule_runs["default"], schedule_runs[variant]
    for name, sensor in (("d32", "hdl32e"), ("d64", "hdl64e")):
        _, i, j = np.intersect1d(d[f"{name}_idx"], v[f"{name}_idx"], return_indices=True)   # the same keypoints
        assert len(i) >= 0.99 * len(d[f"{name}_idx"])
        assert np.array_equal(d[f"{name}_det_nn"][i], v[f"{name}_det_nn"][j])
        rd, rv = d[f"{name}_det_rf"][i], v[f"{name}_det_rf"][j]
        assert np.array_equal(np.isnan(rd), np.isnan(rv))
        ok = ~np.isnan(rd).any(1)
        assert np.abs(rd[ok] - rv[ok]).max() <= 1e-6
        identical = (v[f"{name}_det_bits"][j] == d[f"{name}_det_bits"][i]).all(1).mean()
        print(f"{variant} {name}: {identical:.4%} of {len(i)} descriptors bit-identical to the default")
        pts = synth.make_scan(sensor, 0)
        kp = pts[v[f"{name}_idx"]]
        g = {k: v[f"{name}_det_{k}"] for k in ("bits", "shot", "rf", "nn")}
        which = np.random.default_rng(3).choice(len(kp), 16, replace=False)
        judge(f"{variant} {name}", pts, kp, v[f"{name}_normals"], 3000.0, g, which)
