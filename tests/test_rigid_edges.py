"""The device's rigid fits (icp_fit_kernel, umeyama3) at the shapes and edges where they can go wrong, judged by the
float64 reference of tests/rigid_f64.py with its derived bound -- and, for every case, device == oracle bit for bit.
Each checked fit prints `RATIO <family> rR rt`: its errors as fractions of the bound."""
import numpy as np
import pytest

import rigid_f64 as rf
from test_icp import rigid, rot, scene
from test_ransac import planted
from test_rigid_f64 import assert_rigid, degenerate_icp_cases, lattice_line

f32 = np.float32
pytestmark = pytest.mark.gpu


def same_icp(g, o):
    assert g["iterations"] == o["iterations"] and g["state"] == o["state"]
    assert np.array_equal(g["transform"].view(np.uint32), o["transform"].view(np.uint32)), (g["transform"], o["transform"])
    assert g["mse"] == o["mse"] or (np.isnan(g["mse"]) and np.isnan(o["mse"]))


def report(family, c):
    print(f"RATIO {family} {c['rR']:.4f} {c['rt']:.4f}")


def icp_case(gpu_ctx, oracle, family, src, tgt, pre=None, need_decidable=True):
    """1 and 10 iterations: device == oracle, every transform rigid, every step within the bound"""
    for iters in (1, 10):
        g = gpu_ctx.icp(src, tgt, pre=pre, max_iterations=iters)
        same_icp(g, oracle.icp(src, tgt, pre=pre, max_iterations=iters))
        assert_rigid(g["transform"], f"{family}: device icp, {iters} iterations")
    Ts = [np.eye(4, dtype=f32)] + [gpu_ctx.icp(src, tgt, pre=pre, max_iterations=k)["transform"] for k in range(1, g["iterations"] + 1)]
    ref = rf.icp_f64(src, tgt, pre=pre, iters=g["iterations"], transforms=Ts)
    if need_decidable:
        assert ref["decidable"], family
    if ref["decidable"]:
        for k, c in enumerate(ref["checks"]):
            assert c["ok"], (family, k + 1, c["why"])
            report(family, c)
    return ref


# ---- ICP ----------------------------------------------------------------------------------------------------------------
def test_icp_generic_600x3000(gpu_ctx, oracle):
    src, tgt, _ = scene()
    icp_case(gpu_ctx, oracle, "generic", src, tgt)
    icp_case(gpu_ctx, oracle, "generic", src, tgt, pre=rigid(0.003, (50.0, -20.0, 5.0)))


def test_icp_1e5_sources(gpu_ctx, oracle):
    """10^5 sources: 391 terms per partial sum, the largest fp32 summation error of the suite.  Sources on a fine
    lattice, targets on a coarse one, rotated: no source is near a boundary of its target's Voronoi cell, so every
    nearest target is decidable in fp32 and all ten steps are judged"""
    i, j, k = np.meshgrid(np.arange(50), np.arange(50), np.arange(40), indexing="ij")
    src = (np.c_[i.ravel() * 800.0, j.ravel() * 800.0, k.ravel() * 200.0] - [20000.0, 20000.0, 4000.0] + [37.3, 61.9, 11.7]).astype(f32)
    a, b, c = np.meshgrid(np.arange(10), np.arange(10), np.arange(8), indexing="ij")
    tgt = np.c_[a.ravel() * 4000.0, b.ravel() * 4000.0, c.ravel() * 1000.0] - [18000.0, 18000.0, 3500.0]
    tgt = (tgt @ rot(2e-3).T + [3.0, -2.0, 1.0]).astype(f32)
    ref = icp_case(gpu_ctx, oracle, "generic_1e5", src, tgt)
    assert len(ref["checks"]) == 10


@pytest.mark.parametrize("axis", [2, 0])
def test_icp_mirrored_targets(gpu_ctx, oracle, axis):
    """det Sigma < 0 (the cloud mirrored along its thinnest axis): the proper optimum flips the third axis"""
    rng = np.random.default_rng(12)
    ext = np.full(3, 40000.0)
    ext[axis] = 1500.0
    src = rng.uniform(-1, 1, (80, 3)) * ext
    M = np.ones(3)
    M[axis] = -1.0
    tgt = (src * M + 40.0).astype(f32)
    src = src.astype(f32)
    st = rf.icp_step_f64(src, tgt)
    assert st["fit"]["det"] < 0 and st["fit"]["rank"] == 3
    icp_case(gpu_ctx, oracle, "mirrored", src, tgt)


@pytest.mark.parametrize("flip", [False, True])
def test_icp_planar_sources(gpu_ctx, oracle, flip):
    """rank 2: the completion branch, with det U det V of both signs"""
    rng = np.random.default_rng(5)
    src = rng.uniform(-20000, 20000, (500, 3)).astype(f32)
    src[:, 2] = 0.0
    R = rot(0.01, 0.02) @ (np.diag([1.0, -1.0, -1.0]) if flip else np.eye(3))
    tgt = (src @ (R @ (np.diag([1.0, -1.0, 1.0]) if flip else np.eye(3))).T + [30.0, -20.0, 10.0]).astype(f32)
    st = rf.icp_step_f64(src, tgt)
    assert st["fit"]["rank"] == 2
    icp_case(gpu_ctx, oracle, "planar", src, tgt, need_decidable=False)


@pytest.mark.parametrize("ratio", [0.5e-5, 2e-5])
def test_icp_rank_decision(gpu_ctx, oracle, ratio):
    """s2 / s0 on both sides of the 1e-5 rank threshold: completion and det-sign branches reach the same optimum"""
    g = np.linspace(-3000.0, 3000.0, 7)
    xy = np.array([[x, 0.6 * y] for x in g for y in g])
    c = np.sqrt(ratio * (xy[:, 0] ** 2).mean())
    src = np.concatenate([np.c_[xy, np.full(len(xy), c)], np.c_[xy, np.full(len(xy), -c)]]).astype(f32)
    tgt = (src.astype(np.float64) @ rot(1e-4).T + [2.0, -1.0, 0.5]).astype(f32)
    st = rf.icp_step_f64(src, tgt)
    assert st["fit"]["rank"] == (2 if ratio < 1e-5 else 3)
    assert abs(st["fit"]["sv"][2] / st["fit"]["sv"][0] / ratio - 1.0) < 0.05
    icp_case(gpu_ctx, oracle, "rank_decision", src, tgt)


@pytest.mark.parametrize("case", list(degenerate_icp_cases()))
def test_icp_rank_deficient(gpu_ctx, oracle, case):
    """rank 0 (one target, coincident sources or targets) and rank 1 (two targets, sources on a line): a proper
    rotation, the identity at rank 0, t = dm - R sm"""
    src, tgt = degenerate_icp_cases()[case]
    ref = icp_case(gpu_ctx, oracle, "rank01", src, tgt, need_decidable=False)
    g = gpu_ctx.icp(src, tgt, max_iterations=1)
    if ref["steps"][0]["fit"]["rank"] == 0:
        assert np.array_equal(g["transform"][:3, :3], np.eye(3, dtype=f32))
    c = rf.check_fit(g["transform"][:3, :3], g["transform"][:3, 3], ref["steps"][0]["fit"], rf.fit_bound(ref["steps"][0]["fit"]))
    assert c["ok"], c["why"]


def test_icp_large_offsets(gpu_ctx, oracle):
    """|x| ~ 10^5 mm with a 1 m extent: fp32 centring cancels the most here"""
    rng = np.random.default_rng(31)
    src = (np.array([1.0e5, -0.8e5, 0.3e5]) + rng.uniform(-500, 500, (150, 3))).astype(f32)
    tgt = (src.astype(np.float64) @ rot(2e-3).T + (np.eye(3) - rot(2e-3)) @ [1.0e5, -0.8e5, 0.3e5] + [4.0, -3.0, 2.0]).astype(f32)
    icp_case(gpu_ctx, oracle, "offset", src, tgt)


def test_icp_nan_sources(gpu_ctx, oracle):
    src, tgt, _ = scene(n_src=500, n_extra=2000, seed=41)
    src[::17] = np.nan
    src[5, 1] = np.nan
    icp_case(gpu_ctx, oracle, "nan", src, tgt)


# ---- RANSAC ---------------------------------------------------------------------------------------------------------------
def ransac_case(gpu_ctx, oracle, family, src, tgt, pairs, **kw):
    g = gpu_ctx.ransac(src, tgt, pairs, **kw)
    o = oracle.ransac(src, tgt, pairs, **kw)
    assert g["iterations"] == o["iterations"] and np.array_equal(g["pairs"], o["pairs"])
    assert np.array_equal(g["transform"].view(np.uint32), o["transform"].view(np.uint32))
    assert_rigid(g["transform"], f"{family}: device ransac")
    ref = rf.ransac_f64(src, tgt, pairs, **kw)
    assert ref["decidable"], ref["why"][:3]
    assert g["iterations"] == ref["iterations"] and np.array_equal(g["pairs"], ref["pairs"])
    if ref["iterations"]:
        c = rf.check_ransac_model(g["transform"], ref)
        assert c["ok"], c["why"]
        report(family, c)
    else:
        assert np.array_equal(g["transform"], np.eye(4, dtype=f32))
    return ref


@pytest.mark.parametrize("n,outliers,seed", [(400, 0.4, 0), (2000, 0.7, 1)])
def test_ransac_generic(gpu_ctx, oracle, n, outliers, seed):
    src, tgt, pairs, _, _, _ = planted(n, outliers, seed=seed)
    ransac_case(gpu_ctx, oracle, "ransac", src, tgt, pairs)


@pytest.mark.parametrize("seed,step", [(0, (1000.0, 0.0, 0.0)), (1, (1000.0, 0.0, 0.0)), (0, (1000.0, 500.0, 0.0)), (2, (0.0, 750.0, -250.0))])
def test_ransac_lattice_line(gpu_ctx, oracle, seed, step):
    """every triple exactly collinear: every model has rank 1"""
    src, tgt, pairs = lattice_line(seed=seed, step=step)
    ref = ransac_case(gpu_ctx, oracle, "ransac_rank1", src, tgt, pairs)
    assert ref["fit"]["rank"] == 1


@pytest.mark.parametrize("point", [(100.0, 200.0, 300.0), (1234.567, -89.123, 4.321)])
def test_ransac_lattice_line_coincident_targets(gpu_ctx, oracle, point):
    """targets all on one point: rank 0, R = I -- also where (3 T) / 3 does not round back to T"""
    src, _, pairs = lattice_line()
    tgt = np.tile([point], (len(src), 1)).astype(f32)
    ref = ransac_case(gpu_ctx, oracle, "ransac_rank0", src, tgt, pairs, threshold=30000.0)
    assert ref["fit"]["rank"] == 0
    g = gpu_ctx.ransac(src, tgt, pairs, threshold=30000.0)
    assert np.array_equal(g["transform"][:3, :3], np.eye(3, dtype=f32))


def test_ransac_most_samples_rejected(gpu_ctx, oracle):
    """a tight cluster and a few far points: isSampleGood rejects most draws"""
    rng = np.random.default_rng(7)
    src = np.concatenate([rng.normal(0, 1.0, (170, 3)), rng.uniform(-30000, 30000, (30, 3))]).astype(f32)
    tgt = (src.astype(np.float64) @ rot(0.1).T + [500.0, 0.0, 0.0]).astype(f32)
    pairs = np.stack([np.arange(200), np.arange(200)], 1).astype(np.int32)
    ref = ransac_case(gpu_ctx, oracle, "ransac", src, tgt, pairs)
    assert ref["n_valid"] >= 1


def test_ransac_best_model_under_three_inliers(gpu_ctx, oracle):
    """unrelated pairs and a 10 mm threshold: the best model keeps < 3 inliers, so every pair stays with the identity"""
    rng = np.random.default_rng(9)
    src = rng.uniform(-30000, 30000, (50, 3)).astype(f32)
    tgt = rng.uniform(-30000, 30000, (50, 3)).astype(f32)
    pairs = np.stack([np.arange(50), np.arange(50)], 1).astype(np.int32)
    ref = ransac_case(gpu_ctx, oracle, "ransac", src, tgt, pairs, threshold=10.0)
    assert len(ref["pairs"]) == 50 and ref["iterations"] == 0


# ---- the estimation gate --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["one_target", "one_target_n3", "one_target_n7", "one_target_n63", "coincident_targets_n60", "two_targets"])
def test_gate_rank_deficient_targets(gpu_ctx, oracle, case):
    src, tgt = degenerate_icp_cases()[case]
    T_ref = rigid(0.3, (5000.0, -2000.0, 0.0))
    T_j = (T_ref.astype(np.float64) @ rigid(0.05, (300.0, 0.0, 0.0)).astype(np.float64)).astype(f32)
    g = gpu_ctx.evaluate_estimation(T_j, T_ref, 40, src, tgt, run_icp=True)
    o = oracle.evaluate_estimation(T_j, T_ref, 40, src, tgt, run_icp=True)
    assert np.array_equal(g["T_best"], o["T_best"]) and g["should_update_map"] == o["should_update_map"]
    assert_rigid(g["T_best"], f"evaluate_estimation({case})")
    if case != "two_targets":   # rank 0: ICP adds no rotation to the gated estimate
        T_est = T_j if g["should_update_map"] else T_ref
        assert np.array_equal(g["T_best"][:3, :3], T_est[:3, :3]), (g["T_best"], T_est)
