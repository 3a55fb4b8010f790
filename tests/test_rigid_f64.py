"""CPU checks of the float64 rigid-fit reference (tests/rigid_f64.py) and of its checker: known answers, agreement
with the oracle's ICP and RANSAC on the scenes of test_icp.py / test_ransac.py within the derived bound, the oracle
on rank-deficient inputs, and checker mutations that must fail."""
import numpy as np
import pytest

import rigid_f64 as rf
from test_icp import rot, scene
from test_ransac import planted

f32 = np.float32


def cloud(n=200, scale=(3000.0, 1500.0, 400.0), seed=0):
    return (np.random.default_rng(seed).normal(0, 1, (n, 3)) * scale).astype(f32)


# ---- the reference against known answers -------------------------------------------------------------------------------
def test_known_translation_and_rotation():
    src = cloud()
    fit = rf.umeyama_f64(src, src.astype(np.float64) + [100.0, -50.0, 7.0])
    assert fit["rank"] == 3 and np.allclose(fit["R"], np.eye(3), atol=1e-12) and np.allclose(fit["t"], [100.0, -50.0, 7.0], atol=1e-9)
    R90 = rot(np.pi / 2)
    fit = rf.umeyama_f64(src, src.astype(np.float64) @ R90.T + [1.0, 2.0, 3.0])
    assert np.allclose(fit["R"], R90, atol=1e-12) and np.allclose(fit["t"], [1, 2, 3], atol=1e-9)
    assert fit["opt"] == pytest.approx(fit["sv"].sum(), rel=1e-12)


def test_known_mirror_gives_the_proper_rotation():
    """box corners (diagonal covariance) mirrored in z, the axis of least spread: det Sigma < 0, S(2) = -1,
    R = U diag(1, 1, -1) V^T = I"""
    src = np.array([[x, y, z] for x in (-3000, 3000) for y in (-1500, 1500) for z in (-400, 400)], f32) + f32(50.0)
    dst = src.astype(np.float64) * [1.0, 1.0, -1.0]
    fit = rf.umeyama_f64(src, dst)
    assert fit["rank"] == 3 and fit["det"] < 0
    assert np.allclose(fit["R"], np.eye(3), atol=1e-9) and np.linalg.det(fit["R"]) > 0
    assert fit["opt"] == pytest.approx(fit["sv"][0] + fit["sv"][1] - fit["sv"][2], rel=1e-12)


def test_known_one_target_point():
    src = cloud(50)
    fit = rf.umeyama_f64(src, np.tile([[5.0, 6.0, 7.0]], (50, 1)))
    assert fit["rank"] == 0 and np.array_equal(fit["R"], np.eye(3))
    assert np.allclose(fit["t"], np.array([5.0, 6.0, 7.0]) - src.astype(np.float64).mean(0), atol=1e-9)


@pytest.mark.parametrize("flip", [False, True])
def test_known_planar_cloud_both_signs(flip):
    """planar sources (rank 2); targets rotated, or reflected in the plane -- which a half-turn about x realises"""
    src = cloud(300, (4000.0, 2500.0, 0.0), seed=2)
    R0 = rot(0.3, 0.1)
    M = np.diag([1.0, -1.0, 1.0]) if flip else np.eye(3)
    dst = src.astype(np.float64) @ (R0 @ M).T + [10.0, 20.0, 30.0]
    fit = rf.umeyama_f64(src, dst)
    assert fit["rank"] == 2
    want = R0 @ (np.diag([1.0, -1.0, -1.0]) if flip else np.eye(3))
    assert np.allclose(fit["R"], want, atol=1e-9) and np.linalg.det(fit["R"]) > 0
    assert np.allclose(fit["t"], [10.0, 20.0, 30.0], atol=1e-6)


# ---- the reference against the oracle ------------------------------------------------------------------------------------
ICP_SCENES = [dict(), dict(n_src=400, n_extra=1500, yaw=-0.006, t=(-120.0, 200.0, 10.0), seed=8), dict(n_src=200, n_extra=300)]


@pytest.mark.parametrize("kw", ICP_SCENES)
def test_oracle_icp_step_within_bound(oracle, kw):
    src, tgt, _ = scene(**kw)
    st = rf.icp_step_f64(src, tgt)
    assert (st["gap"] > 1.0).all()
    o = oracle.icp(src, tgt, max_iterations=1)
    c = rf.check_fit(o["transform"][:3, :3], o["transform"][:3, 3], st["fit"], rf.fit_bound(st["fit"]))
    assert c["ok"], c["why"]
    assert abs(o["mse"] - st["mse"]) <= 1e-5 * st["mse"]


def icp_transforms(run, src, tgt, iters=10, pre=None):
    """the 4x4 results of `run` after 0, 1, .., its own iteration count (at most `iters`)"""
    last = run(src, tgt, pre=pre, max_iterations=iters)
    return [np.eye(4, dtype=f32)] + [run(src, tgt, pre=pre, max_iterations=k)["transform"] for k in range(1, last["iterations"] + 1)], last


@pytest.mark.parametrize("kw", ICP_SCENES)
def test_oracle_icp_ten_iterations_within_bound(oracle, kw):
    src, tgt, _ = scene(**kw)
    Ts, last = icp_transforms(oracle.icp, src, tgt)
    assert last["iterations"] >= 5
    ref = rf.icp_f64(src, tgt, iters=last["iterations"], transforms=Ts)
    assert ref["decidable"]
    for k, c in enumerate(ref["checks"]):
        assert c["ok"], (k + 1, c["why"])


@pytest.mark.parametrize("n,outliers,seed", [(400, 0.4, 0), (60, 0.2, 2), (2000, 0.7, 1)])
def test_oracle_ransac_equals_reference(oracle, n, outliers, seed):
    src, tgt, pairs, _, _, _ = planted(n, outliers, seed=seed)
    ref = rf.ransac_f64(src, tgt, pairs)
    o = oracle.ransac(src, tgt, pairs)
    assert ref["decidable"], ref["why"][:3]
    assert o["iterations"] == ref["iterations"] and np.array_equal(o["pairs"], ref["pairs"])
    c = rf.check_ransac_model(o["transform"], ref)
    assert c["ok"], c["why"]


# ---- the oracle on rank-deficient cross-covariances (rank 0 and 1) -----------------------------------------------------
ODD_POINT = np.array([[1234.567, -89.123, 4.321]], f32)


def degenerate_icp_cases():
    rng = np.random.default_rng(11)
    spread = rng.uniform(-3000, 3000, (64, 3)).astype(f32)
    line = np.zeros((64, 3), f32)
    line[:, 0] = np.linspace(-4000, 4000, 64)
    diag = (np.linspace(-1, 1, 64)[:, None] * np.array([[3000.0, -2000.0, 1000.0]]) + [100.0, 200.0, -50.0]).astype(f32)
    return {
        "one_target": (spread[:8], np.array([[700.0, -300.0, 20.0]], f32)),                 # Sigma = 0
        "coincident_sources": (np.tile(spread[:1], (8, 1)), spread),                      # Sigma = 0
        "coincident_targets": (spread, np.tile([[10.0, 20.0, 30.0]], (5, 1)).astype(f32)),  # Sigma = 0
        # n not a power of two and non-dyadic coordinates: the rounded centroid misses the common point, so the computed
        # Sigma is rounding noise with s0 > 0 -- still rank 0
        **{f"one_target_n{n}": (spread[:n], ODD_POINT) for n in (3, 5, 7, 10, 13, 63)},
        **{f"coincident_targets_n{n}": (spread[:n], np.tile(ODD_POINT, (5, 1))) for n in (50, 60, 63)},
        "coincident_sources_n7": (np.tile(ODD_POINT, (7, 1)), spread),
        "two_targets": (spread, np.array([[-2000.0, 0.0, 0.0], [2000.0, 500.0, 0.0]], f32)),  # rank 1
        "line_sources_x": (line, spread),                                                 # rank 1, exact
        "line_sources_diag": (diag, spread),                                              # rank 1 at 1e-5
        "antiparallel_line": (line, (line * [-1.0, 1.0, 1.0])[::-1].copy() + f32(1.0)),
    }


def assert_rigid(T, what):
    R = np.asarray(T, np.float64)[:3, :3]
    assert np.isfinite(R).all(), f"{what}: non-finite R {R.tolist()}"
    orth = np.abs(R.T @ R - np.eye(3)).max()
    assert orth <= 1e-6 and abs(np.linalg.det(R) - 1.0) <= 1e-6, \
        f"{what}: singular or improper R: |R^T R - I| = {orth:.3g}, det {np.linalg.det(R):.3g}, R = {R.round(6).tolist()}"


@pytest.mark.parametrize("case", list(degenerate_icp_cases()))
@pytest.mark.parametrize("iters", [1, 10])
def test_oracle_icp_rank_deficient(oracle, case, iters):
    src, tgt = degenerate_icp_cases()[case]
    o = oracle.icp(src, tgt, max_iterations=iters)
    assert_rigid(o["transform"], f"oracle.icp({case}, {iters})")
    st = rf.icp_step_f64(src, tgt)
    if iters == 1:
        c = rf.check_fit(o["transform"][:3, :3], o["transform"][:3, 3], st["fit"], rf.fit_bound(st["fit"]))
        assert c["ok"], c["why"]
    if st["fit"]["rank"] == 0:
        assert np.array_equal(o["transform"][:3, :3], np.eye(3, dtype=f32)), f"oracle.icp({case}, {iters}): R = {o['transform'][:3, :3].tolist()}"


def lattice_line(n=40, seed=0, step=(1000.0, 0.0, 0.0)):
    """correspondences whose sources lie on one lattice line: every drawn triple is exactly collinear"""
    rng = np.random.default_rng(seed)
    src = (np.arange(n)[:, None] * np.asarray(step) - [20000.0, 0.0, 0.0]).astype(f32)
    tgt = (src.astype(np.float64) @ rot(0.2).T + [300.0, -100.0, 50.0]).astype(f32)
    tgt[rng.random(n) < 0.2] += f32(5000.0)
    return src, tgt, np.stack([np.arange(n), np.arange(n)], 1).astype(np.int32)


def test_oracle_ransac_coincident_odd_targets(oracle):
    """every target on one non-dyadic point: (3 T) / 3 != T in double, Sigma is rounding noise, still rank 0 and R = I"""
    src, _, pairs = lattice_line()
    tgt = np.tile(ODD_POINT, (len(src), 1))
    o = oracle.ransac(src, tgt, pairs, threshold=30000.0)
    assert np.array_equal(o["transform"][:3, :3], np.eye(3, dtype=f32)), o["transform"]
    ref = rf.ransac_f64(src, tgt, pairs, threshold=30000.0)
    assert ref["decidable"] and ref["fit"]["rank"] == 0
    assert o["iterations"] == ref["iterations"] and np.array_equal(o["pairs"], ref["pairs"])
    assert rf.check_ransac_model(o["transform"], ref)["ok"]


@pytest.mark.parametrize("step", [(1000.0, 0.0, 0.0), (1000.0, 500.0, 0.0)])
def test_oracle_ransac_on_a_lattice_line(oracle, step):
    src, tgt, pairs = lattice_line(step=step)
    o = oracle.ransac(src, tgt, pairs)
    assert_rigid(o["transform"], "oracle.ransac(lattice line)")
    ref = rf.ransac_f64(src, tgt, pairs)
    assert ref["decidable"], ref["why"][:3]
    assert o["iterations"] == ref["iterations"] and np.array_equal(o["pairs"], ref["pairs"])
    c = rf.check_ransac_model(o["transform"], ref)
    assert c["ok"], c["why"]


# ---- the checker has teeth -------------------------------------------------------------------------------------------------
def mutations():
    return {
        "transposed": lambda R, t: (R.T, t),
        "third_axis_flipped": lambda R, t: (R @ np.diag([1.0, 1.0, -1.0]), t),
        "rotated_1e-4_rad": lambda R, t: (rot(1e-4) @ R, t),
        "t_off_1mm": lambda R, t: (R, t + [1.0, 0.0, 0.0]),
        "singular": lambda R, t: (R @ np.diag([1.0, 1.0, 0.0]), t),
    }


@pytest.mark.parametrize("name", list(mutations()))
def test_checker_rejects(oracle, name):
    src, tgt, _ = scene(yaw=0.3)
    st = rf.icp_step_f64(src, tgt)
    b = rf.fit_bound(st["fit"])
    o = oracle.icp(src, tgt, max_iterations=1)["transform"].astype(np.float64)
    assert rf.check_fit(o[:3, :3], o[:3, 3], st["fit"], b)["ok"]
    R, t = mutations()[name](o[:3, :3], o[:3, 3])
    c = rf.check_fit(R, t, st["fit"], b)
    assert not c["ok"], (name, b)


def test_checker_requires_the_identity_at_rank_0():
    """rank 0: every R reaches the (zero) objective and satisfies t = dm - R sm, so the checker demands R = I itself"""
    src, tgt = degenerate_icp_cases()["one_target_n7"]
    st = rf.icp_step_f64(src, tgt)
    assert st["fit"]["rank"] == 0
    b = rf.fit_bound(st["fit"])
    fit = st["fit"]
    assert rf.check_fit(np.eye(3), fit["dm"] - fit["sm"], fit, b)["ok"]
    R = rot(1.2566)   # 72 degrees
    c = rf.check_fit(R, fit["dm"] - R @ fit["sm"], fit, b)
    assert not c["ok"] and "identity" in c["why"]


@pytest.mark.parametrize("name", ["third_axis_flipped", "singular", "t_off_1mm"])
def test_checker_rejects_rank_deficient(name):
    """rank <= 1: any proper R with R v0 = u0 passes, an improper or singular one or a wrong t does not"""
    src, tgt = degenerate_icp_cases()["two_targets"]
    st = rf.icp_step_f64(src, tgt)
    assert st["fit"]["rank"] == 1
    b = rf.fit_bound(st["fit"])
    R, t = st["fit"]["R"], st["fit"]["t"]
    assert rf.check_fit(R, t, st["fit"], b)["ok"]
    R2, t2 = mutations()[name](R, t)
    if name != "t_off_1mm":
        t2 = st["fit"]["dm"] - R2 @ st["fit"]["sm"]
    assert not rf.check_fit(R2, t2, st["fit"], b)["ok"], name
