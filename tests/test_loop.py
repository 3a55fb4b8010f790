"""Loop closure in the GPU-resident map: every entry remembers the map update that wrote it, the map keeps the pose of every
update (bshot_gmap_scans), and bshot_detect_loop matches the last scan's reference frame against the entries of older
updates -> RANSAC -> ICP around T_ransac -> a vote for the scan the surviving matches came from -> the loop edge T_rel.

As in test_relocalize.py, a twin context that must give the same descriptors replays the same extractions (the front end
carries the reference's persistent normals from one extraction to the next)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from test_odometry_step import assert_same_report
from test_relocalize import block_coords, distractors, lasers, mul4x4, pose_error, rot_z, same_bits

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "b-shot-slam_b200")

MAP_ENTRIES, MAP_BLOCKS = 1 << 16, 4096


# ---- helpers ----------------------------------------------------------------------------------------------------------------
def step(ctx, L, p):
    return ctx.odometry_step(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p)


def extract(ctx, L, p):
    return ctx.extract_scan(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p.front, vert_init=p.vert_init_rad, lowpt_th=p.lowpt_th,
                            want_cloud=False)


def fresh(bshot, max_targets=1 << 17, max_entries=MAP_ENTRIES):
    ctx = bshot.Context(0, 131072, 1024, max_targets)
    ctx.gmap_create(max_entries, MAP_BLOCKS)
    return ctx


def rigid_inverse(T):
    """odom_math.cuh's rigid_inverse4x4 in fp32: [R^T | -(((r0i t0 + r1i t1) + r2i t2))]"""
    T = np.asarray(T, np.float32)
    o = np.zeros((4, 4), np.float32)
    o[:3, :3] = T[:3, :3].T
    for i in range(3):
        o[i, 3] = -((T[0, i] * T[0, 3] + T[1, i] * T[1, 3]) + T[2, i] * T[2, 3])
    o[3, 3] = np.float32(1.0)
    return o


def vote(tags):
    """the most frequent update index (the lowest on ties) and its count; (-1, 0) without tags"""
    if len(tags) == 0:
        return -1, 0
    u, c = np.unique(np.asarray(tags, np.int64), return_counts=True)
    best = int(np.argmax(c))   # np.unique sorts: the first maximum is the lowest index
    return int(u[best]), int(c[best])


def in_cube(xyz, T, rng):
    """gm_cube around T's translation (fp32 (p -+ range) / 10 m, rounded half away) against the entries' block coordinates"""
    p = np.asarray(T, np.float32)[:3, 3]
    lo = block_coords((p - np.float32(rng)).reshape(1, 3))[0]
    hi = block_coords((p + np.float32(rng)).reshape(1, 3))[0]
    b = block_coords(xyz)
    return np.all((b >= lo) & (b <= hi), axis=1)


def host_detect(twin, f, xyzr, desc, tags, poses, scan, lp):
    """bshot_detect_loop as host calls on a twin context: candidate filter, match_mutual, ransac, cube filter, icp, mul4x4,
    vote, rigid inverse.  f = the twin's extraction of the scan (its reference frame)"""
    cand = (tags.astype(np.int64) + lp.min_gap) <= scan
    cx, cd, ct = xyzr[cand, :3], desc[cand], tags[cand]
    pairs = twin.match_mutual(f["bits"], cd)[0] if len(cd) else np.empty((0, 2), np.int32)
    rs = twin.ransac(f["kp_xyz"], cx, pairs, lp.ransac_iterations, lp.inlier_threshold)
    T_r = rs["transform"]
    n_icp, icp_it, T_loop = 0, 0, T_r
    if lp.run_icp:
        tx = cx[in_cube(cx, T_r, lp.map_range)]
        ic = twin.icp(f["kp_xyz"], tx, pre=T_r, max_iterations=10)
        n_icp, icp_it, T_loop = len(tx), ic["iterations"], mul4x4(ic["transform"], T_r)
    inl = rs["pairs"]
    match, votes = vote(ct[inl[:, 1]]) if len(inl) else (-1, 0)
    T_rel = mul4x4(rigid_inverse(poses[match]), T_loop) if match >= 0 else np.eye(4, dtype=np.float32)
    return dict(T_loop=T_loop, T_ransac=T_r, T_rel=T_rel, pose=poses[scan], n_candidates=int(cand.sum()), n_icp_targets=n_icp, scan=scan,
                match_scan=match, votes=votes, n_keypoints=len(f["bits"]), n_pairs=len(pairs), n_inliers=len(inl),
                ransac_iterations=rs["iterations"], icp_iterations=icp_it, accepted=int(len(inl) >= lp.min_inliers))


LOOP_INTS = ("n_candidates", "n_icp_targets", "scan", "match_scan", "votes", "n_keypoints", "n_pairs", "n_inliers", "ransac_iterations",
             "icp_iterations", "accepted")


def assert_same_loop(a, b, where=""):
    for key in ("T_loop", "T_ransac", "T_rel", "pose"):
        assert same_bits(np.asarray(a[key], np.float32), np.asarray(b[key], np.float32)), (where, key, a[key], b[key])
    for key in LOOP_INTS:
        assert int(a[key]) == int(b[key]), (where, key, a[key], b[key])


def pose_T(x, y, yaw_deg):
    T = np.eye(4)
    T[:3, :3] = rot_z(yaw_deg)
    T[:3, 3] = [x, y, 0.0]
    return T


# ---- CPU --------------------------------------------------------------------------------------------------------------------
def test_loop_symbols_exported(bshot):
    L = bshot.lib()
    for s in ("bshot_gmap_scans", "bshot_loop_params_default", "bshot_detect_loop"):
        assert s in bshot.EXPORTS and hasattr(L, s), s
    R = bshot.LoopReport
    assert (R.T_loop.offset, R.T_ransac.offset, R.T_rel.offset, R.pose.offset) == (0, 64, 128, 192)
    assert (R.n_candidates.offset, R.n_icp_targets.offset, R.scan.offset, R.accepted.offset) == (256, 264, 272, 304)
    assert ctypes.sizeof(R) == 312
    P = bshot.LoopParams
    assert (P.min_gap.offset, P.inlier_threshold.offset, P.run_icp.offset, ctypes.sizeof(P)) == (0, 12, 20, 24)


def test_loop_params_default(bshot):
    p = bshot.loop_params_default()
    assert (p.min_gap, p.min_inliers, p.ransac_iterations, p.inlier_threshold, p.map_range, p.run_icp) == (100, 15, 2000, 1500.0, 100000.0, 1)
    assert bshot.loop_params_default(min_gap=7, run_icp=0).min_gap == 7
    with pytest.raises(AttributeError):
        bshot.loop_params_default(no_such_field=1)


def test_rigid_inverse_replica_against_float64():
    """the fp32 replica of the rigid inverse and of T_rel = T_j^-1 * T_loop, against float64 inverses: within a few ulp of
    the translations' magnitude"""
    rng = np.random.default_rng(3)
    for _ in range(200):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        w, x, y, z = q
        R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                      [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                      [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
        Tj, Tl = np.eye(4), np.eye(4)
        Tj[:3, :3], Tj[:3, 3] = R, rng.uniform(-1e5, 1e5, 3)
        Tl[:3, :3], Tl[:3, 3] = rot_z(rng.uniform(-180, 180)) @ R, rng.uniform(-1e5, 1e5, 3)
        Tj32, Tl32 = Tj.astype(np.float32), Tl.astype(np.float32)
        inv = rigid_inverse(Tj32)
        ref = np.linalg.inv(Tj32.astype(np.float64))
        scale = np.abs(Tj32[:3, 3]).sum()
        assert np.abs(inv[:3, :3] - ref[:3, :3]).max() <= 2e-7
        assert np.abs(inv[:3, 3] - ref[:3, 3]).max() <= 4e-7 * scale
        assert np.array_equal(inv[3], [0, 0, 0, 1])
        rel = mul4x4(inv, Tl32)
        rel_ref = ref @ Tl32.astype(np.float64)
        assert np.abs(rel[:3, :3] - rel_ref[:3, :3]).max() <= 1e-6
        assert np.abs(rel[:3, 3] - rel_ref[:3, 3]).max() <= 1e-6 * (scale + np.abs(Tl32[:3, 3]).sum())
    assert vote([]) == (-1, 0) and vote([4, 2, 4, 2, 9]) == (2, 2) and vote([7, 7, 1]) == (7, 2)


@pytest.fixture(scope="module")
def loop_shim_binary(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("loop_shim") / "host_shim_loop_test")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror", os.path.join(ROOT, "tests", "host_shim_loop_test.cpp"),
                           "-o", out, "-L", PKG, "-lbshot_b200", f"-Wl,-rpath,{PKG}"])
    return out


def _write_rotations(tmp_path, synth, frames):
    L0 = synth.make_lasers("hdl32e", frames[0])
    ring = str(tmp_path / "ring.bin")
    np.ascontiguousarray(L0["ring_deg"], np.float64).tofile(ring)
    rec = np.dtype([("az", "<f8"), ("ve", "<f8"), ("di", "<u2")])
    paths = []
    for f in frames:
        L = synth.make_lasers("hdl32e", f)
        a = np.empty(len(L["azimuth"]), rec)
        a["az"], a["ve"], a["di"] = L["azimuth"], L["vertical"], L["distance"]
        paths.append(str(tmp_path / f"rot{f}.bin"))
        a.tofile(paths[-1])
    return ring, paths


def test_loop_shim_fails_loudly_without_gpu(loop_shim_binary, tmp_path, synth):
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    ring, paths = _write_rotations(tmp_path, synth, [0])
    r = subprocess.run([loop_shim_binary, ring, str(tmp_path / "out.bin"), "1", paths[0]], capture_output=True, text=True)
    assert r.returncode == 1 and "no CUDA device" in r.stdout


# ---- GPU: tags and trajectory ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_tags_and_trajectory(bshot, synth):
    """after every step u: an entry whose (position, seg-ratio, descriptor) is new carries tag u, every other entry keeps
    its tag; the trajectory is the steps' poses bit for bit.  After an import: every tag 0, the trajectory one identity"""
    p = bshot.odom_default_params(top_k=600)
    with fresh(bshot) as a:
        prev = {}
        poses = []
        for u in range(12):
            r = step(a, lasers(synth, u), p)
            poses.append(r["pose"])
            x, d = a.gmap_export()
            tags, traj = a.gmap_scans()
            assert len(tags) == len(x) and len(traj) == u + 1, u
            cur = {}
            for e in range(len(x)):
                key = x[e, :3].tobytes()
                val = x[e, 3:].tobytes() + d[e].tobytes()
                cur[key] = (val, int(tags[e]))
                if key in prev and prev[key][0] == val:
                    assert tags[e] == prev[key][1], (u, e)
                else:
                    assert tags[e] == u, (u, e, tags[e])
            prev = cur
            for v in range(u + 1):
                assert same_bits(traj[v], poses[v]), (u, v)
        assert len(set(int(t) for t in tags)) > 3   # entries of many scans survive
        x, d = a.gmap_export()
        with fresh(bshot) as b:
            b.gmap_import(x, d)
            tags, traj = b.gmap_scans()
            assert len(tags) == len(x) and not tags.any()
            assert len(traj) == 1 and same_bits(traj[0], np.eye(4, dtype=np.float32))
            # the next step is update 1: its new entries carry 1, its pose is the trajectory's second entry
            s = step(b, lasers(synth, 0), p)
            tags, traj = b.gmap_scans()
            assert len(traj) == 2 and same_bits(traj[1], s["pose"]) and set(np.unique(tags)) <= {0, 1}
            b.gmap_reset()
            tags, traj = b.gmap_scans()
            assert len(tags) == 0 and len(traj) == 0


# ---- GPU: the detection is its stages -------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("run_icp", [1, 0])
def test_detect_equals_host_stages(bshot, synth, run_icp):
    """12 rotations; the last one against the entries of updates <= 7, on every matcher kind: every report equal to the
    host composition on a twin that replayed the extractions, bit for bit, and identical across matchers"""
    p = bshot.odom_default_params(top_k=600)
    lp = bshot.loop_params_default(min_gap=4, run_icp=run_icp)
    n = 12
    with fresh(bshot) as dev, fresh(bshot) as twin:
        for k in range(n):
            step(dev, lasers(synth, k), p)
            f = extract(twin, lasers(synth, k), p)
        x, d = dev.gmap_export()
        tags, poses = dev.gmap_scans()
        assert len(poses) == n
        reports = []
        for matcher in (-1, 0, 1, 2, 3):
            dev.set_matcher(matcher)
            twin.set_matcher(matcher)
            rd = dev.detect_loop(lp)
            rh = host_detect(twin, f, x, d, tags, poses, n - 1, lp)
            assert_same_loop(rd, rh, matcher)
            reports.append(rd)
        for r in reports[1:]:
            assert_same_loop(r, reports[0])
        r = reports[0]
        print(f"scan {r['scan']}: {r['n_candidates']} candidates, {r['n_inliers']} inliers, match {r['match_scan']} ({r['votes']} votes)")
        assert r["accepted"] == 1 and 0 <= r["match_scan"] <= n - 1 - lp.min_gap and r["n_candidates"] < len(x)


# ---- GPU: revisits --------------------------------------------------------------------------------------------------------
def _route():
    """out along x (40 scans, 500 mm apart, no yaw); a turn onto a lane 1.5 m to the side with the yaw ramped 5 degrees a
    scan to 20; back along that lane in 500 mm steps.  (x, y, yaw) per scan"""
    out = [(500.0 * k, 0.0, 0.0) for k in range(40)]
    turn = [(19500.0 - 250.0 * r, 375.0 * r, 5.0 * r) for r in range(1, 5)]
    back = [(18500.0 - 500.0 * r, 1500.0, 20.0) for r in range(1, 36)]
    return out, turn, back


@pytest.mark.gpu
def test_revisits_are_found(bshot, synth):
    """the way back, 1.5 m beside the way out and yawed by 20 degrees, is closed against the way out.  min_gap = 39 leaves
    every scan of the turn and of the way back out of the candidates of the scans asserted here, so a match can only be a
    scan of the way out (asserted).  Ground truth in the map frame (the first scan's sensor frame): scan at (x, y) with
    yaw, z = 0.

    For the scans of the way back within the first 8 m of the street (the way out's scans there are at least 39
    updates older): accepted, match_scan on the way out, T_loop within TOL of the truth and closer to it than the
    odometry's own pose (T_loop measures the drift).  T_rel = T_j^-1 * T_loop carries the odometry's error of T_j as
    well: with e_j its translation error, th_j its rotation error and el / rl T_loop's, T_rel's translation error is at
    most el + e_j + th_j * |t_rel| and its rotation error at most rl + th_j; that bound (plus 1 mm / 0.01 degree of
    rounding) is asserted.  Scans farther out are printed, not asserted: their place on the way out is less than 39
    updates older, so its entries are not candidates.
    Measured on one NVIDIA B200: 28-46 inliers; T_loop 19-187 mm / 0.03-1.18 deg from the truth while the odometry
    was 0.97-1.42 m off.  TOL = 300 mm / 2 deg leaves about 1.6x."""
    TOL_MM, TOL_DEG = 300.0, 2.0
    out, turn, back = _route()
    route = out + turn + back
    p = bshot.odom_default_params(top_k=600)
    lp = bshot.loop_params_default(min_gap=39)
    rows = []
    with fresh(bshot) as ctx:
        for i, (x, y, yaw) in enumerate(route):
            s = ctx.odometry_step_cloud(synth.make_scan("hdl32e", i, pos=[x, y, 0.0], yaw_deg=yaw), p)
            if i < len(out) + len(turn):
                continue
            d = ctx.detect_loop(lp)
            T_i = pose_T(x, y, yaw)
            el = pose_error(d["T_loop"], T_i[:3, :3], T_i[:3, 3])
            eo = pose_error(s["pose"], T_i[:3, :3], T_i[:3, 3])
            j = d["match_scan"]
            print(f"scan {i} at ({x:.0f}, {y:.0f}, {yaw:.0f} deg): accepted {d['accepted']}, match {j} ({d['votes']} of {d['n_inliers']} inliers); "
                  f"T_loop {el[0]:.1f} mm {el[1]:.3f} deg, odometry {eo[0]:.1f} mm {eo[1]:.3f} deg")
            if x <= 8000.0:
                rows.append((i, d, el, eo))
        _, traj = ctx.gmap_scans()
    print(f"{len(rows)} revisits asserted; worst T_loop {max(r[2][0] for r in rows):.1f} mm {max(r[2][1] for r in rows):.3f} deg, "
          f"best odometry {min(r[3][0] for r in rows):.1f} mm")
    assert len(rows) == 15
    for i, d, el, eo in rows:
        j = d["match_scan"]
        assert d["scan"] == i and d["accepted"] == 1 and 0 <= j < len(out), (i, d)
        assert el[0] < TOL_MM and el[1] < TOL_DEG and el[0] < eo[0], (i, el, eo)
        T_j = pose_T(*route[j])
        rel = np.linalg.inv(T_j) @ pose_T(*route[i])
        er = pose_error(d["T_rel"], rel[:3, :3], rel[:3, 3])
        ej = pose_error(traj[j], T_j[:3, :3], T_j[:3, 3])
        bound_mm = el[0] + ej[0] + np.radians(ej[1]) * np.linalg.norm(rel[:3, 3]) + 1.0
        assert er[0] <= bound_mm and er[1] <= el[1] + ej[1] + 0.01, (i, j, er, el, ej, bound_mm)


@pytest.mark.gpu
def test_drift_is_measured(bshot, synth):
    """session B restores session A's map and starts, without relocalising, 5 m down the street: its first step leaves it
    at the identity, and the detection against the imported map (update 0) measures the 5 m it is off.
    Measured on one NVIDIA B200: 82 inliers, T_rel 40.8 mm / 0.51 deg from the truth; the tolerances leave about 2x."""
    TOL_MM, TOL_DEG = 300.0, 1.0
    p = bshot.odom_default_params(top_k=600)
    with fresh(bshot) as a:
        for k in range(12):
            a.odometry_step_cloud(synth.make_scan("hdl32e", k, pos=[500.0 * k, 0.0, 0.0], yaw_deg=0.0), p)
        x, d = a.gmap_export()
    with fresh(bshot) as b:
        b.gmap_import(x, d)
        s = b.odometry_step_cloud(synth.make_scan("hdl32e", 10, pos=[5000.0, 0.0, 0.0], yaw_deg=0.0), p)
        assert s["was_initial"] == 1
        r = b.detect_loop(bshot.loop_params_default(min_gap=1))
        dt, da = pose_error(r["T_rel"], np.eye(3), [5000.0, 0.0, 0.0])
        print(f"drift: accepted {r['accepted']}, match {r['match_scan']}, {r['n_inliers']} inliers, T_rel off by {dt:.1f} mm {da:.3f} deg")
        assert r["scan"] == 1 and r["match_scan"] == 0 and r["accepted"] == 1 and r["votes"] == r["n_inliers"]
        assert dt < TOL_MM and da < TOL_DEG, (dt, da)
        assert same_bits(r["pose"], s["pose"]) and same_bits(r["T_rel"], r["T_loop"])   # T_0 is the identity


# ---- GPU: negatives and errors --------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_negatives_and_errors(bshot, synth):
    p = bshot.odom_default_params(top_k=600)
    lp = bshot.loop_params_default

    def code(ctx, params=None):
        with pytest.raises(bshot.BshotError) as e:
            ctx.detect_loop(params)
        return e.value.code

    with bshot.Context(0, 131072, 1024, 1 << 16) as c:
        assert code(c) == bshot.E_STATE   # no map
    with fresh(bshot) as a:
        assert code(a) == bshot.E_STATE   # no step yet
        for k in range(3):
            step(a, lasers(synth, k), p)
        r = a.detect_loop(lp(min_gap=100))   # no candidates
        assert r["accepted"] == 0 and r["n_candidates"] == 0 and r["match_scan"] == -1 and r["scan"] == 2
        for bad in (lp(min_gap=0), lp(min_gap=-3), lp(min_inliers=2), lp(ransac_iterations=0), lp(inlier_threshold=0.0)):
            assert code(a, bad) == bshot.E_INVALID
        x, d = a.gmap_export()
        f = a.extract_frame(synth.make_scan("hdl32e", 3), p.front)
        assert a.detect_loop(lp(min_gap=1))["scan"] == 2   # an extraction changes neither the map nor the reference frame
        a.frame_commit()
        assert code(a) == bshot.E_STATE
        step(a, lasers(synth, 3), p)
        a.gmap_update_from_frame(np.eye(4, dtype=np.float32)[:3])
        assert code(a) == bshot.E_STATE
        step(a, lasers(synth, 4), p)
        a.gmap_add(f["kp_xyz"], f["seg_ratio"], f["bits"])
        assert code(a) == bshot.E_STATE
        step(a, lasers(synth, 5), p)
        a.gmap_import(x, d)
        assert code(a) == bshot.E_STATE
        step(a, lasers(synth, 6), p)
        assert a.detect_loop(lp(min_gap=1))["scan"] == 1
        a.gmap_reset()
        assert code(a) == bshot.E_STATE
        step(a, lasers(synth, 7), p)
        a.odometry_reset()
        assert code(a) == bshot.E_STATE
    # a map of distractors only
    with fresh(bshot) as b:
        dx, dd = distractors(synth, 20000)
        b.gmap_import(dx, dd)
        step(b, lasers(synth, 0), p)
        r = b.detect_loop(lp(min_gap=1))
        print(f"distractors: {r['n_candidates']} candidates, {r['n_pairs']} pairs, {r['n_inliers']} inliers")
        assert r["n_candidates"] == 20000 and r["accepted"] == 0
    # more ICP targets than max_targets
    with fresh(bshot) as a:
        for k in range(12):
            step(a, lasers(synth, k), p)
        x, d = a.gmap_export()
    assert len(x) > 1024
    with fresh(bshot, max_targets=1024) as c:
        c.gmap_import(x, d)
        step(c, lasers(synth, 6), p)   # INITIAL: the frame against itself, no map targets
        tags0, traj0 = c.gmap_scans()
        assert code(c, lp(min_gap=1)) == bshot.E_CAPACITY
        r = c.detect_loop(lp(min_gap=1, run_icp=0))
        assert r["accepted"] == 1 and r["n_icp_targets"] == 0 and r["icp_iterations"] == 0 and same_bits(r["T_loop"], r["T_ransac"])
        tags1, traj1 = c.gmap_scans()
        assert np.array_equal(tags0, tags1) and same_bits(traj0, traj1)


# ---- GPU: read only ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_detection_is_read_only(bshot, synth):
    """detections on every matcher leave the map, the tags, the trajectory and the next steps as a twin has them that
    never detected"""
    p = bshot.odom_default_params(top_k=600)
    with fresh(bshot) as a, fresh(bshot) as t:
        for k in range(8):
            assert_same_report(step(a, lasers(synth, k), p), step(t, lasers(synth, k), p), k)
        x0, d0 = a.gmap_export()
        g0, p0 = a.gmap_scans()
        for matcher in (-1, 0, 2):
            a.set_matcher(matcher)
            assert a.detect_loop(bshot.loop_params_default(min_gap=3))["accepted"] == 1
            a.detect_loop(bshot.loop_params_default(min_gap=3, run_icp=0))
        a.set_matcher(-1)
        x1, d1 = a.gmap_export()
        g1, p1 = a.gmap_scans()
        assert same_bits(x0, x1) and np.array_equal(d0, d1) and np.array_equal(g0, g1) and same_bits(p0, p1)
        for k in (8, 9):
            assert_same_report(step(a, lasers(synth, k), p), step(t, lasers(synth, k), p), k)
        xa, da = a.gmap_export()
        xt, dt = t.gmap_export()
        assert same_bits(xa, xt) and np.array_equal(da, dt)
        assert np.array_equal(a.gmap_scans()[0], t.gmap_scans()[0])


# ---- GPU: C++ shim ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_device_odometry_loop_shim_equals_python(bshot, synth, loop_shim_binary, tmp_path):
    frames = list(range(7))
    ring, paths = _write_rotations(tmp_path, synth, frames)
    out = str(tmp_path / "out.bin")
    r = subprocess.run([loop_shim_binary, ring, out, "3"] + paths, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = np.fromfile(out, np.uint8)
    p = bshot.odom_default_params()
    with bshot.Context(0, 131072, 1024, 1 << 16) as c:
        c.gmap_create(1 << 16, 4096)
        for k in frames:
            step(c, lasers(synth, k), p)
        lr = c.detect_loop(bshot.loop_params_default(min_gap=3))
        _, traj = c.gmap_scans()
    assert raw.size == 128 + 24 + 64 * len(traj)
    assert same_bits(raw[:64].view(np.float32).reshape(4, 4), lr["T_loop"])
    assert same_bits(raw[64:128].view(np.float32).reshape(4, 4), lr["T_rel"])
    assert list(raw[128:152].view(np.int32)) == [lr["scan"], lr["match_scan"], lr["votes"], lr["n_inliers"], lr["accepted"], lr["n_candidates"]]
    assert same_bits(raw[152:].view(np.float32).reshape(-1, 4, 4), traj)
