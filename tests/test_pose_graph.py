"""bshot_optimize_trajectory: the trajectory's pose graph optimised on the device in float64, judged against the float64
reference of tests/pose_graph_f64.py (LM with exact sparse solves) through its checker."""
import ctypes
import os
import re

import numpy as np
import pytest

from pose_graph_f64 import Graph, check_optimum, jr_inv, so3_exp, so3_log
from test_loop import _route, fresh, pose_T
from test_reanchor import rot_xyz
from test_relocalize import pose_error, same_bits

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def random_walk(n, seed, step_mm=500.0, yaw_deg=2.0):
    rng = np.random.default_rng(seed)
    T = np.eye(4)
    out = [T.copy()]
    for _ in range(n - 1):
        D = np.eye(4)
        D[:3, :3] = rot_xyz(*np.radians(rng.normal(0.0, [0.2, 0.2, yaw_deg])))
        D[:3, 3] = [step_mm, rng.normal(0.0, 50.0), rng.normal(0.0, 10.0)]
        T = T @ D
        out.append(T.copy())
    return np.asarray(out)


def synthetic(n, n_loops, seed):
    """truth, a drifted trajectory (the truth's increments with a yaw bias and noise, scaled so that the whole chain drifts
    by a few degrees whatever n is) and loop edges measured from the truth with 30 mm / 0.2 deg noise"""
    rng = np.random.default_rng(seed + 100)
    truth = random_walk(n, seed)
    drift = [truth[0].copy()]
    k = min(1.0, np.sqrt(100.0 / n))
    for u in range(1, n):
        D = np.linalg.inv(truth[u - 1]) @ truth[u]
        E = np.eye(4)
        E[:3, :3] = rot_xyz(*np.radians(rng.normal(0.0, 0.05 * k, 3) + [0.0, 0.0, min(0.05, 5.0 / n)]))
        E[:3, 3] = rng.normal(0.0, 10.0 * k, 3)
        drift.append(drift[-1] @ D @ E)
    drift = np.asarray(drift).astype(np.float32)
    drift[:, 3] = [0, 0, 0, 1]
    loops = []
    for _ in range(n_loops):
        a, b = sorted(rng.choice(n, 2, replace=False))
        M = np.linalg.inv(truth[a]) @ truth[b]
        N = np.eye(4)
        N[:3, :3] = rot_xyz(*np.radians(rng.normal(0.0, 0.2, 3)))
        N[:3, 3] = rng.normal(0.0, 30.0, 3)
        T = (M @ N).astype(np.float32)
        T[3] = [0, 0, 0, 1]
        loops.append((int(a), int(b), T))
    return truth, drift, loops


def graph_context(bshot, poses):
    """a context whose map has one update per pose (gmap_add of one entry with that pose): its trajectory is poses"""
    ctx = bshot.Context(0, 16384, 1024, 4096)
    ctx.gmap_create(max(2 * len(poses), 1024), len(poses) // 10 + 64)
    one = np.zeros((1, 3), np.float32)
    desc = np.zeros((1, 6), np.uint64)
    for P in poses:
        ctx.gmap_add(one, np.ones(1, np.float32), desc, np.asarray(P, np.float32)[:3])
    return ctx


# ---- CPU --------------------------------------------------------------------------------------------------------------------
def _decl_fields(struct):
    h = open(os.path.join(ROOT, "include", "bshot_b200.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (struct, struct), h, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return re.findall(r"\b([A-Za-z_]+)(?:\[\d+\])?\s*[,;]", body)


def test_exports_layout_and_defaults(bshot):
    L = bshot.lib()
    for s in ("bshot_graph_params_default", "bshot_optimize_trajectory"):
        assert s in bshot.EXPORTS and hasattr(L, s), s
    assert [f.rstrip("_") for f, _ in bshot.GraphEdge._fields_] == _decl_fields("bshot_graph_edge")
    assert [f for f, _ in bshot.GraphParams._fields_] == _decl_fields("bshot_graph_params")
    assert [f for f, _ in bshot.GraphReport._fields_] == _decl_fields("bshot_graph_report")
    assert (bshot.GraphEdge.T.offset, ctypes.sizeof(bshot.GraphEdge)) == (8, 72)
    P = bshot.GraphParams
    assert (P.max_iterations.offset, P.grad_tolerance.offset, P.cg_tolerance.offset, ctypes.sizeof(P)) == (16, 24, 40, 48)
    R = bshot.GraphReport
    assert (R.status.offset, R.cost_initial.offset, R.grad_inf_final.offset, ctypes.sizeof(R)) == (16, 24, 40, 48)
    p = bshot.graph_params_default()
    assert (p.odom_sigma_mm, round(p.odom_sigma_deg, 6), p.loop_sigma_mm, p.loop_sigma_deg) == (20.0, 0.1, 100.0, 1.0)
    assert (p.max_iterations, p.max_cg_iterations, p.grad_tolerance, p.step_tolerance, p.cg_tolerance) == (50, 2000, 1e-6, 1e-9, 1e-10)
    assert bshot.graph_params_default(max_iterations=3).max_iterations == 3


def test_reference_jacobians_match_central_differences():
    truth, drift, loops = synthetic(6, 3, seed=2)
    g = Graph(drift, loops)
    R, t = g.R0.copy(), g.t0.copy()
    R[1:] = R[1:] @ so3_exp(np.random.default_rng(0).normal(0, 0.01, (5, 3)))
    r0, Ja, Jb = g.jacobians(R, t)
    h = 1e-6
    for node, J, sel in ((g.ea, Ja, 0), (g.eb, Jb, 1)):
        for k in range(6):
            # per edge, perturb the node of this side alone
            for e in range(len(node)):
                rp, rm = [], []
                for s, acc in ((1.0, rp), (-1.0, rm)):
                    R2, t2 = R.copy(), t.copy()
                    i = node[e]
                    if k < 3:
                        t2[i, k] += s * h
                    else:
                        w = np.zeros(3)
                        w[k - 3] = s * h
                        R2[i] = R[i] @ so3_exp(w)
                    rt, rr, _ = g.residuals(R2, t2)
                    acc.append(np.concatenate([rt[e], rr[e]]))
                fd = (rp[0] - rm[0]) / (2 * h)
                scale = max(1.0, np.abs(J[e][:, k]).max())
                assert np.abs(fd - J[e][:, k]).max() <= 1e-5 * scale, (sel, e, k, fd, J[e][:, k])
    # the series branches agree with the closed forms across their switch
    for th in (0.5e-4, 2e-4):
        w = np.array([th, 0.0, 0.0])
        assert np.allclose(so3_log(so3_exp(w)), w, rtol=1e-9, atol=1e-15)
        assert np.allclose(jr_inv(w), jr_inv(w * (1 + 1e-9)), atol=1e-9)


def test_reference_recovers_a_consistent_graph():
    """measurements taken from a known trajectory, the solve started 0.5 m / 1 deg away: the known trajectory comes back to
    float64 rounding"""
    truth = random_walk(30, seed=4)
    loops = [(0, 29, (np.linalg.inv(truth[0]) @ truth[29]).astype(np.float32)), (5, 20, (np.linalg.inv(truth[5]) @ truth[20]).astype(np.float32))]
    g = Graph(truth.astype(np.float32), loops)
    T32 = truth.astype(np.float32).astype(np.float64)
    rng = np.random.default_rng(1)
    g.R0[1:] = g.R0[1:] @ so3_exp(rng.normal(0, np.radians(1.0), (29, 3)))
    g.t0[1:] += rng.normal(0, 500.0, (29, 3))
    # loop measurements from the fp32 poses are consistent with them up to fp32 rounding of T
    res = g.solve(max_iterations=100, grad_tolerance=1e-12, step_tolerance=0.0)
    assert np.abs(res["t"] - T32[:, :3, 3]).max() < 1e-3
    assert np.abs(res["R"] - T32[:, :3, :3]).max() < 1e-7


def test_checker_rejects_a_moved_optimum():
    truth, drift, loops = synthetic(40, 5, seed=7)
    g = Graph(drift, loops)
    ref = g.solve(max_iterations=100, grad_tolerance=1e-10, step_tolerance=0.0)
    P = np.tile(np.eye(4), (g.n, 1, 1))
    P[:, :3, :3], P[:, :3, 3] = ref["R"], ref["t"]
    check_optimum(g, ref, P.astype(np.float32), 1e-12)
    moved = P.copy()
    moved[17, 0, 3] += 1.0
    with pytest.raises(AssertionError):
        check_optimum(g, ref, moved.astype(np.float32), 1e-12)
    moved = P.copy()
    moved[23, :3, :3] = moved[23, :3, :3] @ so3_exp(np.array([0.0, 1e-4, 0.0]))
    with pytest.raises(AssertionError):
        check_optimum(g, ref, moved.astype(np.float32), 1e-12)


# ---- GPU --------------------------------------------------------------------------------------------------------------------
CHAINS = [(2, 1), (50, 1), (50, 10), (1000, 10), (1000, 100), (10000, 10), (10000, 100)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,n_loops", CHAINS)
def test_synthetic_chains_reach_the_reference_optimum(bshot, n, n_loops):
    truth, drift, loops = synthetic(n, n_loops, seed=n + n_loops)
    with graph_context(bshot, drift) as ctx:
        p = bshot.graph_params_default(max_iterations=100, grad_tolerance=1e-7)
        out = ctx.optimize_trajectory(loops, p)
    g = Graph(drift, loops)
    ref = g.solve(max_iterations=100, grad_tolerance=1e-9, step_tolerance=1e-12)
    dist, bound = check_optimum(g, ref, out["poses"], out["grad_inf_final"])
    et0 = np.abs(drift[:, :3, 3] - truth[:, :3, 3]).max()
    et1 = np.abs(out["poses"][:, :3, 3] - truth[:, :3, 3]).max()
    print(f"n {n} L {n_loops}: {out['iterations']} LM, {out['cg_iterations']} CG (12 L + 1 = {12 * n_loops + 1} a solve), status {out['status']}, "
          f"cost {out['cost_initial']:.4g} -> {out['cost_final']:.4g} (reference {ref['cost']:.4g}), |g| {out['grad_inf_final']:.3g}; "
          f"distance {dist:.3g} <= {bound:.3g}; max drift {et0:.0f} -> {et1:.0f} mm")
    assert out["status"] in (1, 2, 3) and out["cost_final"] <= out["cost_initial"]
    assert out["cost_final"] <= ref["cost"] * (1 + 1e-6) + 1e-9
    assert same_bits(out["poses"][0], drift[0])


@pytest.mark.gpu
def test_no_loops_deterministic_read_only_and_errors(bshot):
    truth, drift, loops = synthetic(200, 20, seed=3)
    with graph_context(bshot, drift) as ctx:
        out = ctx.optimize_trajectory([])
        assert out["iterations"] == 0 and out["status"] == 1 and same_bits(out["poses"], drift)
        x0, d0 = ctx.gmap_export()
        s0 = ctx.gmap_scans()
        a = ctx.optimize_trajectory(loops)
        b = ctx.optimize_trajectory(loops)
        assert same_bits(a["poses"], b["poses"]) and np.array_equal(a["loop_cost"].view(np.uint64), b["loop_cost"].view(np.uint64))
        assert (a["iterations"], a["cg_iterations"], a["cost_final"]) == (b["iterations"], b["cg_iterations"], b["cost_final"])
        x1, d1 = ctx.gmap_export()
        s1 = ctx.gmap_scans()
        assert same_bits(x0, x1) and np.array_equal(d0, d1) and np.array_equal(s0[0], s1[0]) and same_bits(s0[1], s1[1])
        # one wrong loop edge: the largest loop cost
        bad = list(loops)
        T = np.eye(4, dtype=np.float32)
        T[:3, 3] = [3000.0, -2000.0, 0.0]
        bad.append((10, 150, T))
        c = ctx.optimize_trajectory(bad)
        assert int(np.argmax(c["loop_cost"])) == len(bad) - 1, c["loop_cost"]

        def code(lp, params=None):
            with pytest.raises(bshot.BshotError) as e:
                ctx.optimize_trajectory(lp, params)
            return e.value.code
        eye = np.eye(4, dtype=np.float32)
        for lp in ([(0, 200, eye)], [(-1, 3, eye)], [(4, 4, eye)], [(1, 2, eye * np.float32(1.1))], [(1, 2, np.full((4, 4), np.nan, np.float32))]):
            assert code(lp) == bshot.E_INVALID
        for kw in (dict(odom_sigma_mm=0.0), dict(loop_sigma_deg=-1.0), dict(max_iterations=-1), dict(max_cg_iterations=-1), dict(grad_tolerance=-1.0),
                   dict(step_tolerance=-1.0), dict(cg_tolerance=-1.0)):
            assert code(loops, bshot.graph_params_default(**kw)) == bshot.E_INVALID
        p12 = np.empty((10, 3, 4), np.float32)
        r = bshot.GraphReport()
        rc = bshot.lib().bshot_optimize_trajectory(ctx.h, None, 0, ctypes.byref(bshot.graph_params_default()), p12.ctypes.data_as(ctypes.c_void_p), 10, None,
                                                   ctypes.byref(r))
        assert rc == bshot.E_CAPACITY
    with bshot.Context(0, 1024, 64, 64) as c:
        with pytest.raises(bshot.BshotError) as e:
            c.optimize_trajectory([])
        assert e.value.code == bshot.E_STATE
    with graph_context(bshot, drift[:1]) as c:
        out = c.optimize_trajectory([])
        assert out["iterations"] == 0 and same_bits(out["poses"], drift[:1])


@pytest.mark.gpu
def test_detect_optimise_reanchor_on_the_street(bshot, synth):
    """the street of test_loop.py with min_gap = 39: the accepted detections of the way back up to 3.5 m down the street
    become loop edges; optimise, then re-anchor.  (a) every way-back scan within the first 8 m is closer to the truth than
    the odometry had it, and within TOL_MM; (b) detect_loop right after on the same scan measures a drift well below the
    one before; (c) the next steps stay closer to the truth than a twin's that did not close the loop.
    Measured on one NVIDIA B200 (1000 W limit): 10 loop edges, 5 LM iterations, 52 CG iterations; the way back within 8 m
    62-187 mm from the truth against the odometry's 974-1271 mm; detected drift 1306 -> 227 mm; the next three steps
    226-309 mm against the twin's 1271-1346 mm.  TOL_MM = 400 leaves about 2x."""
    TOL_MM = 400.0
    out, turn, back = _route()
    route = out + turn + back
    n = len(out) + len(turn) + 30   # the last scan at x = 3.5 m
    p = bshot.odom_default_params(top_k=600)
    lp = bshot.loop_params_default(min_gap=39)

    def scan(i):
        x, y, yaw = route[i]
        return synth.make_scan("hdl32e", i, pos=[x, y, 0.0], yaw_deg=yaw)

    def drift(d):
        D = np.linalg.inv(np.asarray(d["pose"], np.float64)) @ np.asarray(d["T_loop"], np.float64)
        return float(np.linalg.norm(D[:3, 3]))

    with fresh(bshot) as a, fresh(bshot) as t:
        loops, odo = [], {}
        for i in range(n):
            cloud = scan(i)
            s = a.odometry_step_cloud(cloud, p)
            t.odometry_step_cloud(cloud, p)
            odo[i] = s["pose"]
            if i >= len(out) + len(turn):
                d = a.detect_loop(lp)
                if d["accepted"]:
                    loops.append(d)
        d_before = a.detect_loop(lp)
        res = a.optimize_trajectory(loops)
        pose = a.gmap_reanchor(res["poses"])
        d_after = a.detect_loop(lp)
        rows = []
        for i in range(len(out) + len(turn), n):
            T = pose_T(*route[i])
            eo = pose_error(odo[i], T[:3, :3], T[:3, 3])[0]
            ec = pose_error(res["poses"][i], T[:3, :3], T[:3, 3])[0]
            if route[i][0] <= 8000.0:
                rows.append((i, eo, ec))
        print(f"{len(loops)} loop edges; {res['iterations']} LM, {res['cg_iterations']} CG, status {res['status']}, cost {res['cost_initial']:.4g} -> "
              f"{res['cost_final']:.4g}; way back within 8 m: odometry {min(r[1] for r in rows):.0f}-{max(r[1] for r in rows):.0f} mm, "
              f"optimised {min(r[2] for r in rows):.0f}-{max(r[2] for r in rows):.0f} mm; drift {drift(d_before):.0f} -> {drift(d_after):.0f} mm")
        assert len(loops) >= 5 and rows
        for i, eo, ec in rows:
            assert ec < eo and ec < TOL_MM, (i, eo, ec)
        assert same_bits(pose[:3], res["poses"][-1][:3])
        assert drift(d_after) < 0.5 * drift(d_before), (drift(d_before), drift(d_after))
        for i in range(n, n + 3):
            T, cloud = pose_T(*route[i]), scan(i)
            ea = pose_error(a.odometry_step_cloud(cloud, p)["pose"], T[:3, :3], T[:3, 3])[0]
            et = pose_error(t.odometry_step_cloud(cloud, p)["pose"], T[:3, :3], T[:3, 3])[0]
            print(f"scan {i}: closed {ea:.0f} mm, twin {et:.0f} mm")
            assert ea < et, (i, ea, et)
