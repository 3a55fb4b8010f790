"""Re-anchoring the GPU-resident map to a corrected trajectory (bshot_gmap_reanchor): every entry moves by the correction
C_u = T'_u * T_u^-1 of the update u that wrote it, snapped to the 10 mm lattice; the map is rebuilt in export order; the
trajectory becomes the corrected one and the odometry's pose follows its last update.

The numpy replica below restates the move in fp32 (odom_math.cuh's mul4x4 / rigid_inverse4x4, gm_prepare_kernel's
transform, createKeypoint's truncation) and the rebuild as a stable regroup by block; the GPU tests hold the device to it
bit for bit."""
import os
import subprocess

import numpy as np
import pytest

from test_loop import _route, _write_rotations, fresh, lasers, pose_T, rigid_inverse, step
from test_odometry_step import assert_same_report
from test_relocalize import block_coords, mul4x4, pose_error, same_bits

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "b-shot-slam_b200")


# ---- the replica ------------------------------------------------------------------------------------------------------------
def transform_rn(C, xyz):
    """gm_prepare_kernel's R p + T: ((c0 x + c1 y) + c2 z) + c3 per row, every operation rounded to fp32"""
    C = np.asarray(C, np.float32)
    p = np.asarray(xyz, np.float32)
    out = np.empty_like(p)
    for r in range(3):
        out[:, r] = ((C[r, 0] * p[:, 0] + C[r, 1] * p[:, 1]) + C[r, 2] * p[:, 2]) + C[r, 3]
    return out


def snap(v):
    """Keypoint::createKeypoint: int(trunc(v / 10)) * 10, in fp32"""
    q = np.asarray(v, np.float32) / np.float32(10.0)
    return (np.trunc(q).astype(np.int64) * 10).astype(np.float32)


def changed_updates(traj, new):
    old12 = np.ascontiguousarray(np.asarray(traj, np.float32)[:, :3, :]).reshape(len(traj), 12)
    new12 = np.ascontiguousarray(np.asarray(new, np.float32)[:, :3, :]).reshape(len(new), 12)
    return np.any(old12.view(np.uint32) != new12.view(np.uint32), axis=1)


def correction(T_old, T_new):
    return mul4x4(T_new, rigid_inverse(T_old))


def replica_reanchor(xyzr, desc, tags, traj, new, pose):
    """-> (xyzr, desc, tags) in the new export order and the odometry's new pose"""
    chg = changed_updates(traj, new)
    moved = np.array(xyzr, np.float32, copy=True)
    for u in np.flatnonzero(chg):
        sel = tags == u
        if sel.any():
            moved[sel, :3] = snap(transform_rn(correction(traj[u], new[u]), moved[sel, :3]))
    b = block_coords(moved[:, :3])
    order = np.lexsort((b[:, 2], b[:, 1], b[:, 0]))   # stable: export order survives inside a block
    last = len(traj) - 1
    T_last = np.asarray(traj[last], np.float32)
    if not chg[last]:
        pose_new = np.asarray(pose, np.float32)
    elif same_bits(np.asarray(pose, np.float32)[:3], T_last[:3]):
        pose_new = np.asarray(new[last], np.float32).copy()
        pose_new[3] = [0, 0, 0, 1]
    else:
        pose_new = mul4x4(correction(traj[last], new[last]), pose)
    return moved[order], np.asarray(desc)[order], np.asarray(tags)[order], pose_new


def rot_xyz(ax, ay, az):
    cx, sx, cy, sy, cz, sz = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay), np.cos(az), np.sin(az)
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    return Rz @ Ry @ Rx


def corrected(traj, seed=5, deg=0.3, mm=60.0, keep=(0,)):
    """traj moved by a random walk of small corrections, computed in float64 and rounded to fp32; updates in keep stay"""
    rng = np.random.default_rng(seed)
    out = np.array(traj, np.float32, copy=True)
    D = np.eye(4)
    for u in range(len(traj)):
        step_D = np.eye(4)
        step_D[:3, :3] = rot_xyz(*np.radians(rng.normal(0.0, deg, 3)))
        step_D[:3, 3] = rng.normal(0.0, mm, 3)
        D = step_D @ D
        if u not in keep:
            out[u] = (D @ np.asarray(traj[u], np.float64)).astype(np.float32)
            out[u, 3] = [0, 0, 0, 1]
    return out


# ---- CPU --------------------------------------------------------------------------------------------------------------------
def test_reanchor_exported(bshot):
    assert "bshot_gmap_reanchor" in bshot.EXPORTS and hasattr(bshot.lib(), "bshot_gmap_reanchor")


def test_replica_move_and_regroup():
    """the replica on cases with known answers: exact dyadic motions, the truncating snap, the stable regroup by block, and
    the pose rule"""
    assert list(snap([15.0, -15.0, 9.99, -9.99, 20.0, 123456.7])) == [10.0, -10.0, 0.0, -0.0, 20.0, 123450.0]
    # a quarter turn about z and an integer shift are exact in fp32
    T_old = np.eye(4, dtype=np.float32)
    T_new = np.eye(4, dtype=np.float32)
    T_new[:3, :3] = [[0, -1, 0], [1, 0, 0], [0, 0, 1]]
    T_new[:3, 3] = [20000.0, 0.0, 30.0]
    p = np.array([[1000.0, 2000.0, 0.0], [4990.0, -30.0, 10.0]], np.float32)
    assert same_bits(transform_rn(correction(T_old, T_new), p), np.array([[18000.0, 1000.0, 30.0], [20030.0, 4990.0, 40.0]], np.float32))
    # three entries of update 1 in one block, one of update 0; update 1 moves 20 m along x, past update 0's entry
    xyzr = np.array([[100, 0, 0, 0.1], [200, 0, 0, 0.2], [300, 0, 0, 0.3], [12000, 0, 0, 0.4]], np.float32)
    desc = np.arange(24, dtype=np.uint64).reshape(4, 6)
    tags = np.array([1, 1, 1, 0], np.uint32)
    traj = np.stack([np.eye(4, dtype=np.float32)] * 2)
    new = traj.copy()
    new[1, 0, 3] = 20000.0
    x, d, t, pose = replica_reanchor(xyzr, desc, tags, traj, new, traj[1])
    assert list(x[:, 0]) == [12000.0, 20100.0, 20200.0, 20300.0] and list(x[:, 3]) == list(np.float32([0.4, 0.1, 0.2, 0.3]))
    assert list(t) == [0, 1, 1, 1] and np.array_equal(d[1:], desc[:3])
    assert same_bits(pose, new[1])
    # the pose is not the last update's: it moves by that update's correction
    off = np.eye(4, dtype=np.float32)
    off[:3, 3] = [5.0, 6.0, 7.0]
    assert same_bits(replica_reanchor(xyzr, desc, tags, traj, new, off)[3][:3, 3], np.float32([20005.0, 6.0, 7.0]))
    # nothing changed: the export order and the pose as they were
    x, d, t, pose = replica_reanchor(xyzr, desc, tags, traj, traj.copy(), off)
    b = block_coords(xyzr[:, :3])
    assert same_bits(x, xyzr[np.lexsort((b[:, 2], b[:, 1], b[:, 0]))]) and same_bits(pose, off)


def test_corrections_are_rigid_enough():
    """the test trajectories pass the call's rigidity check (max |R^T R - I| <= 1e-3, det R > 0)"""
    traj = np.stack([pose_T(500.0 * k, 10.0 * k, 2.0 * k).astype(np.float32) for k in range(30)])
    new = corrected(traj)
    for T in new.astype(np.float64):
        assert np.abs(T[:3, :3].T @ T[:3, :3] - np.eye(3)).max() < 1e-5 and np.linalg.det(T[:3, :3]) > 0
    assert same_bits(new[0], traj[0]) and changed_updates(traj, new)[1:].all()


@pytest.fixture(scope="module")
def reanchor_shim_binary(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("reanchor_shim") / "host_shim_reanchor_test")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror", os.path.join(ROOT, "tests", "host_shim_reanchor_test.cpp"),
                           "-o", out, "-L", PKG, "-lbshot_b200", f"-Wl,-rpath,{PKG}"])
    return out


def test_reanchor_shim_fails_loudly_without_gpu(reanchor_shim_binary, tmp_path, synth):
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    ring, paths = _write_rotations(tmp_path, synth, [0])
    r = subprocess.run([reanchor_shim_binary, ring, str(tmp_path / "out.bin"), "1", paths[0], paths[0]], capture_output=True, text=True)
    assert r.returncode == 1 and "no CUDA device" in r.stdout


# ---- GPU --------------------------------------------------------------------------------------------------------------------
def snapshot(ctx):
    x, d = ctx.gmap_export()
    tags, traj = ctx.gmap_scans()
    return x, d, tags, traj, ctx.gmap_size()


def assert_same_snapshot(a, b, where=""):
    assert same_bits(a[0], b[0]) and np.array_equal(a[1], b[1]), (where, "export")
    assert np.array_equal(a[2], b[2]), (where, "tags")
    assert same_bits(a[3], b[3]), (where, "trajectory")
    assert tuple(a[4]) == tuple(b[4]), (where, "size", a[4], b[4])


@pytest.mark.gpu
def test_unchanged_trajectory_is_a_no_op(bshot, synth):
    """re-anchoring with the current trajectory: the pose, export, tags, trajectory, size and the next steps are bit for bit
    those of a twin that never re-anchored; loop detection runs on the same scan right after"""
    p = bshot.odom_default_params(top_k=600)
    with fresh(bshot) as a, fresh(bshot) as t:
        for k in range(8):
            r = step(a, lasers(synth, k), p)
            assert_same_report(r, step(t, lasers(synth, k), p), k)
        before = snapshot(a)
        pose = a.gmap_reanchor(before[3])
        assert same_bits(pose, r["pose"])
        assert_same_snapshot(snapshot(a), before)
        assert a.detect_loop(bshot.loop_params_default(min_gap=3))["scan"] == 7
        for k in (8, 9):
            assert_same_report(step(a, lasers(synth, k), p), step(t, lasers(synth, k), p), k)
        assert_same_snapshot(snapshot(a), snapshot(t))


@pytest.mark.gpu
def test_moved_map_equals_the_replica(bshot, synth):
    """a random-walk correction of every update but 0: export and tags equal the replica bit for bit, a twin's import of
    the replica's arrays holds the same map, the trajectory is the input, the pose is T'_{n-1}; then detection and steps run.
    Second round: after gmap_add with a pose of its own the odometry's pose is not the last update's, and it moves by
    C_{n-1}"""
    p = bshot.odom_default_params(top_k=600)
    with fresh(bshot) as a:
        for k in range(10):
            r = step(a, lasers(synth, k), p)
        x0, d0, tags0, traj0, _ = snapshot(a)
        new = corrected(traj0)
        rx, rd, rt, rpose = replica_reanchor(x0, d0, tags0, traj0, new, r["pose"])
        pose = a.gmap_reanchor(new)
        x1, d1, tags1, traj1, size1 = snapshot(a)
        moved = int(np.any(x1[:, :3] != x0[:, :3], axis=1).sum())
        print(f"{len(x0)} entries, {moved} at a new position")
        assert moved > len(x0) // 2
        assert same_bits(x1, rx) and np.array_equal(d1, rd) and np.array_equal(tags1, rt)
        assert same_bits(traj1, new) and same_bits(pose, rpose) and same_bits(pose, new[-1])
        assert size1[0] == len(x0)
        with fresh(bshot) as b:
            b.gmap_import(rx, rd)
            xb, db = b.gmap_export()
            assert same_bits(xb, x1) and np.array_equal(db, d1)
        d = a.detect_loop(bshot.loop_params_default(min_gap=3))
        assert d["scan"] == 9 and same_bits(d["pose"], new[-1])
        s = step(a, lasers(synth, 10), p)
        assert s["n_inliers"] >= 15
        # the pose is not the last update's
        f = a.extract_frame(synth.make_scan("hdl32e", 3), p.front)
        P = pose_T(300.0, -200.0, 4.0).astype(np.float32)
        a.gmap_add(f["kp_xyz"], f["seg_ratio"], f["bits"], P[:3])
        x0, d0, tags0, traj0, _ = snapshot(a)
        assert same_bits(traj0[-1], P)
        new = corrected(traj0, seed=9)
        rx, rd, rt, rpose = replica_reanchor(x0, d0, tags0, traj0, new, s["pose"])
        pose = a.gmap_reanchor(new)
        x1, d1, tags1, traj1, _ = snapshot(a)
        assert same_bits(x1, rx) and np.array_equal(d1, rd) and np.array_equal(tags1, rt) and same_bits(traj1, new)
        assert same_bits(pose, rpose) and not same_bits(pose, new[-1])


@pytest.mark.gpu
def test_capacity_error_changes_nothing(bshot, synth):
    """100 updates of 10 entries, all in one block (32 chunks of the 97 the map holds); a correction that puts each update
    20 m further along x needs 100 chunks: BSHOT_E_CAPACITY, and the map, tags, trajectory, size and pose are as before.
    A correction that fits then succeeds"""
    rng = np.random.default_rng(4)
    lat = np.stack(np.meshgrid(*[np.arange(10) * 1000.0 - 4500.0] * 3, indexing="ij"), -1).reshape(-1, 3).astype(np.float32)
    desc = synth.random_descriptors(1000, seed=4)
    with bshot.Context(0, 16384, 1024, 4096) as c:
        c.gmap_create(1024, 1)
        for u in range(100):
            c.gmap_add(lat[10 * u:10 * u + 10], rng.uniform(0, 1, 10).astype(np.float32), desc[10 * u:10 * u + 10])
        before = snapshot(c)
        assert len(before[0]) == 1000 and len(before[3]) == 100
        pose0 = c.gmap_reanchor(before[3])
        spread = before[3].copy()
        spread[:, 0, 3] = 20000.0 * np.arange(100)
        with pytest.raises(bshot.BshotError) as e:
            c.gmap_reanchor(spread)
        assert e.value.code == bshot.E_CAPACITY
        assert_same_snapshot(snapshot(c), before)
        assert same_bits(c.gmap_reanchor(before[3]), pose0)
        fits = before[3].copy()
        fits[:, 0, 3] = 20000.0 * (np.arange(100) // 50)   # two blocks
        c.gmap_reanchor(fits)
        x, d, tags, traj, _ = snapshot(c)
        rx, rd, rt, _ = replica_reanchor(*before[:4], fits, pose0)
        assert same_bits(x, rx) and np.array_equal(d, rd) and np.array_equal(tags, rt) and same_bits(traj, fits)


@pytest.mark.gpu
def test_invalid_inputs_change_nothing(bshot, synth):
    p = bshot.odom_default_params(top_k=600)

    def code(ctx, poses):
        with pytest.raises(bshot.BshotError) as e:
            ctx.gmap_reanchor(poses)
        return e.value.code

    with bshot.Context(0, 131072, 1024, 1 << 16) as c:
        assert code(c, np.zeros((0, 4, 4), np.float32)) == bshot.E_STATE   # no map
    with fresh(bshot) as a:
        assert same_bits(a.gmap_reanchor(np.zeros((0, 4, 4), np.float32)), np.eye(4, dtype=np.float32))   # no update: nothing to move
        for k in range(4):
            step(a, lasers(synth, k), p)
        before = snapshot(a)
        traj = before[3]
        bad = []
        bad.append(traj[:3])                               # fewer poses than updates
        bad.append(np.concatenate([traj, traj[:1]]))       # more
        for v in (np.nan, np.inf):
            t = traj.copy()
            t[2, 1, 3] = v
            bad.append(t)
        t = traj.copy()
        t[1, :3, :3] *= np.float32(1.01)                   # not orthonormal
        bad.append(t)
        t = traj.copy()
        t[3, :3, 2] *= np.float32(-1.0)                    # a reflection
        bad.append(t)
        for b in bad:
            assert code(a, b) == bshot.E_INVALID
            assert_same_snapshot(snapshot(a), before)
        # within the tolerance: accepted
        t = traj.copy()
        t[1, :3, :3] *= np.float32(1.0004)
        a.gmap_reanchor(t)


@pytest.mark.gpu
def test_true_trajectory_closes_the_loop(bshot, synth):
    """the street of test_loop.py: out along x, turn, back 1.5 m beside the way out, stopped 7.5 m down the street, where
    the way out's scans are loop candidates (min_gap = 39) and the odometry is about 1 m off.  Re-anchoring to the true trajectory (what an ideal back end would return) must
    (a) put the pose within 10 mm / 0.05 deg of the truth, (b) make detect_loop on the same scan measure a drift
    |T_i^-1 T_loop| well below the one it measured before, and (c) keep the next four steps closer to the truth than a
    twin's that did not re-anchor, and within TOL_STEP_MM.
    Measured on one NVIDIA B200 (1000 W limit): the odometry 974 mm / 0.77 deg off before; detected drift 915 mm before,
    95.5 mm after; the next steps 107-136 mm off against the twin's 1099-1132 mm.  TOL_DRIFT_MM = 200 and TOL_STEP_MM =
    250 leave about 2x."""
    TOL_DRIFT_MM, TOL_STEP_MM = 200.0, 250.0
    out, turn, back = _route()
    route = out + turn + back
    n = len(out) + len(turn) + 22   # the last scan at x = 7.5 m
    p = bshot.odom_default_params(top_k=600)
    lp = bshot.loop_params_default(min_gap=39)

    def scan(i):
        x, y, yaw = route[i]
        return synth.make_scan("hdl32e", i, pos=[x, y, 0.0], yaw_deg=yaw)

    def drift(d):
        D = np.linalg.inv(np.asarray(d["pose"], np.float64)) @ np.asarray(d["T_loop"], np.float64)
        return float(np.linalg.norm(D[:3, 3]))

    with fresh(bshot) as a, fresh(bshot) as t:
        for i in range(n):
            cloud = scan(i)
            s = a.odometry_step_cloud(cloud, p)
            assert_same_report(s, t.odometry_step_cloud(cloud, p), i)
        T_i = pose_T(*route[n - 1])
        e_before = pose_error(s["pose"], T_i[:3, :3], T_i[:3, 3])
        d_before = a.detect_loop(lp)
        truth = np.stack([pose_T(*route[u]) for u in range(n)]).astype(np.float32)
        pose = a.gmap_reanchor(truth)
        e_after = pose_error(pose, T_i[:3, :3], T_i[:3, 3])
        d_after = a.detect_loop(lp)
        print(f"scan {n - 1}: odometry {e_before[0]:.1f} mm {e_before[1]:.3f} deg off -> {e_after[0]:.2f} mm {e_after[1]:.4f} deg; "
              f"detected drift {drift(d_before):.1f} mm (accepted {d_before['accepted']}) -> {drift(d_after):.1f} mm (accepted {d_after['accepted']})")
        assert e_before[0] > 500.0
        assert e_after[0] < 10.0 and e_after[1] < 0.05
        assert d_before["accepted"] == 1 and d_after["accepted"] == 1
        assert drift(d_before) > 900.0 and drift(d_after) < TOL_DRIFT_MM, (drift(d_before), drift(d_after))
        for i in range(n, n + 4):
            T, cloud = pose_T(*route[i]), scan(i)
            ea = pose_error(a.odometry_step_cloud(cloud, p)["pose"], T[:3, :3], T[:3, 3])
            et = pose_error(t.odometry_step_cloud(cloud, p)["pose"], T[:3, :3], T[:3, 3])
            print(f"scan {i}: re-anchored {ea[0]:.1f} mm {ea[1]:.3f} deg, twin {et[0]:.1f} mm {et[1]:.3f} deg")
            assert ea[0] < et[0] and ea[0] < TOL_STEP_MM, (i, ea, et)


@pytest.mark.gpu
def test_device_odometry_reanchor_shim_equals_python(bshot, synth, reanchor_shim_binary, tmp_path):
    """DeviceOdometry: steps, detectLoop, reanchor to trajectory() with update u shifted by 10 u mm along x, one more
    step; the same through the Python calls gives the same bits"""
    frames = list(range(7))
    ring, paths = _write_rotations(tmp_path, synth, frames)
    out = str(tmp_path / "out.bin")
    r = subprocess.run([reanchor_shim_binary, ring, out, "3"] + paths, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    print(r.stdout)
    raw = np.fromfile(out, np.uint8)
    p = bshot.odom_default_params()
    with bshot.Context(0, 131072, 1024, 1 << 16) as c:
        c.gmap_create(1 << 16, 4096)
        for k in frames[:-1]:
            step(c, lasers(synth, k), p)
        lr = c.detect_loop(bshot.loop_params_default(min_gap=3))
        _, traj = c.gmap_scans()
        new = traj.copy()
        new[:, 0, 3] += np.float32(10.0) * np.arange(len(traj), dtype=np.float32)
        pose = c.gmap_reanchor(new)
        s = step(c, lasers(synth, frames[-1]), p)
        _, traj2 = c.gmap_scans()
    assert raw.size == 4 + 64 * 2 + 64 * len(traj2)
    assert int(raw[:4].view(np.int32)[0]) == lr["accepted"]
    assert same_bits(raw[4:68].view(np.float32).reshape(4, 4), pose)
    assert same_bits(raw[68:132].view(np.float32).reshape(4, 4), s["pose"])
    assert same_bits(raw[132:].view(np.float32).reshape(-1, 4, 4), traj2)
