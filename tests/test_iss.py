"""ISS keypoints (pcl::ISSKeypoint3D as issKpDetection calls it, src/lidar_odometry.cpp:447-461) and keypoint
repeatability (kpEvaluation, :392-445).  CPU: known answers of the oracle and an independent numpy / scipy restatement.
GPU: bshot_detect_iss / bshot_kp_repeatability against the oracle, no side effects on the frame path, ISS keypoints
through B-SHOT, and the host shim's issKpDetection / kpEvaluation."""
import os
import struct
import subprocess

import numpy as np
import pytest
from scipy.spatial import cKDTree

import iss_oracle  # CPU restatement of ISS and of the repeatability measure (tests/iss_oracle.cpp)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "b-shot-slam_b200")
DEFAULTS = dict(salient_radius=60.0, non_max_radius=40.0, gamma_21=0.975, gamma_32=0.975, min_neighbors=5)


def _corner(seed, n=12, ext=100.0, noise=1.0):
    """three perpendicular 100 mm square grids meeting at the origin, gaussian noise on every coordinate"""
    rng = np.random.default_rng(seed)
    g = np.linspace(0.0, ext, n)
    A, B = np.meshgrid(g, g)
    pts = []
    for ax in range(3):
        P = np.zeros((A.size, 3))
        c = [k for k in range(3) if k != ax]
        P[:, c[0]], P[:, c[1]] = A.ravel(), B.ravel()
        pts.append(P)
    P = np.unique(np.concatenate(pts), axis=0)
    return (P + rng.normal(0.0, noise, P.shape)).astype(np.float32)


def _plane(seed, n=30, step=10.0, z_noise=0.0, xy_noise=2.0):
    rng = np.random.default_rng(seed)
    g = np.arange(n) * step
    A, B = np.meshgrid(g, g)
    P = np.stack([A.ravel(), B.ravel(), np.zeros(A.size)], 1)
    P[:, :2] += rng.normal(0.0, xy_noise, (P.shape[0], 2))
    P[:, 2] += rng.normal(0.0, z_noise, P.shape[0]) if z_noise else 0.0
    return P.astype(np.float32)


def _fp32_sqd(q, pts):
    """flann::L2_Simple in fp32: ((dx*dx) + dy*dy) + dz*dz, no contraction (numpy float32 arithmetic)"""
    d = (pts - q).astype(np.float32)
    return (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]


def _numpy_iss(xyz, salient_radius, non_max_radius, gamma_21, gamma_32, min_neighbors):
    """independent restatement: cKDTree with a slightly larger ball, the fp32 `<` filter, numpy.linalg.eigvalsh"""
    n = len(xyz)
    fin = np.isfinite(xyz).all(1)
    idx_fin = np.nonzero(fin)[0]
    tree = cKDTree(xyz[fin].astype(np.float64))

    def ball(i, r):
        r2 = np.float32(np.float64(r) * np.float64(r))
        cand = idx_fin[tree.query_ball_point(xyz[i].astype(np.float64), r * (1 + 1e-5) + 1e-3)]
        return cand[_fp32_sqd(xyz[i], xyz[cand]) < r2]

    eigs = np.zeros((n, 3))
    third = np.zeros(n)
    for i in idx_fin:
        nb = ball(i, salient_radius)
        if len(nb) < min_neighbors:
            continue
        d = xyz[nb].astype(np.float64) - xyz[i].astype(np.float64)
        w = np.linalg.eigvalsh(d.T @ d)
        eigs[i] = w[::-1]
        e1, e2, e3 = eigs[i]
        if np.isfinite(eigs[i]).all() and e3 >= 0 and e2 / e1 < gamma_21 and e3 / e2 < gamma_32:
            third[i] = e3
    kp = [i for i in idx_fin if third[i] > 0 and len(nb := ball(i, non_max_radius)) >= min_neighbors
          and not (third[nb] > third[i]).any()]
    return np.array(kp, np.int64), eigs


def _ambiguous(i, xyz, eigs, prm, tree):
    """the decision of point i cannot be told apart at 1e-9 relative precision: a ratio within 1e-9 of its threshold,
    lambda3 below 1e-12 lambda1, or a neighbour (within r_nm) whose lambda3 is within 1e-9 relative of its own or whose
    own saliency is such a near-tie"""
    def near_tie(j):
        e1, e2, e3 = eigs[j]
        with np.errstate(divide="ignore", invalid="ignore"):
            return (abs(e2 / e1 - prm["gamma_21"]) < 1e-9 or abs(e3 / e2 - prm["gamma_32"]) < 1e-9 or abs(e3) < 1e-12 * e1)
    if near_tie(i):
        return True
    l3 = eigs[i, 2]
    for j in tree.query_ball_point(xyz[i].astype(np.float64), prm["non_max_radius"] * (1 + 1e-5) + 1e-3):
        if j != i and (abs(eigs[j, 2] - l3) <= 1e-9 * abs(l3) or near_tie(j)):
            return True
    return False


def _compare_keypoints(got, want, xyz, eigs, prm, what):
    got, want = set(int(i) for i in got), set(int(i) for i in want)
    diff = sorted(got ^ want)
    if diff:
        print(f"{what}: {len(diff)} keypoint decisions differ: {diff[:20]}")
    fin = np.isfinite(xyz).all(1)
    tree = cKDTree(np.where(fin[:, None], xyz, 1e30).astype(np.float64))
    assert all(_ambiguous(i, xyz, eigs, prm, tree) for i in diff), (what, diff)
    assert len(diff) <= max(2, int(0.001 * len(want))), (what, diff)


def _compare_eigs(got, want, what):
    tol = 1e-9 * np.abs(want[:, :1])
    bad = np.abs(got - want) > tol
    assert not bad.any(), (what, np.nonzero(bad.any(1))[0][:10])


# ---- CPU: the restatement (tests/iss_oracle.cpp) -------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(4))
def test_cpu_iss_corner_gives_one_keypoint_at_the_corner(oracle, seed):
    P = _corner(seed)
    kp = iss_oracle.iss(oracle.Cloud(P), **DEFAULTS)
    assert len(kp) == 1
    # the vertex itself is not salient (three-fold symmetry: lambda2 == lambda3); the keypoint is the corner point with
    # the most pronounced third eigenvalue, well inside the non-max radius of the vertex
    assert np.linalg.norm(P[kp[0]]) < 30.0


def test_cpu_iss_plane_gives_none(oracle):
    # points jittered within the plane z = 0: lambda3 is exactly 0 everywhere, no point can be a keypoint
    assert len(iss_oracle.iss(oracle.Cloud(_plane(1, xy_noise=2.0)), **DEFAULTS)) == 0
    # noise across the plane: lambda3 > 0, but away from the border (where the ball is cut) lambda2/lambda1 stays above
    # gamma_21, so nothing is salient there
    P = _plane(2, n=40, xy_noise=0.0, z_noise=1.0)
    kp = iss_oracle.iss(oracle.Cloud(P), **DEFAULTS)
    inner = (P[:, :2] > 100.0).all(1) & (P[:, :2] < 290.0).all(1)
    assert inner.sum() > 200 and not inner[kp].any()


def test_cpu_iss_too_few_neighbours(oracle):
    P = _corner(0)[:4]
    kp, eigs = iss_oracle.iss(oracle.Cloud(P), **DEFAULTS, want_eigs=True)
    assert len(kp) == 0 and not eigs.any()                       # fewer than min_neighbors: zero scatter matrix
    assert len(iss_oracle.iss(oracle.Cloud(np.zeros((0, 3), np.float32)), **DEFAULTS)) == 0


def test_cpu_iss_nonfinite_points(oracle):
    P = _corner(3)
    bad = np.array([[np.nan, 0, 0], [0, np.inf, 0], [1.0, 2.0, -np.inf]], np.float32)
    at = [0, 50, 200]
    Q = np.insert(P, at, bad, axis=0)
    keep = np.isfinite(Q).all(1)
    kp, eigs = iss_oracle.iss(oracle.Cloud(P), **DEFAULTS, want_eigs=True)
    kq, eq = iss_oracle.iss(oracle.Cloud(Q), **DEFAULTS, want_eigs=True)
    orig = np.nonzero(keep)[0]
    assert np.array_equal(kq, orig[kp])                         # never a keypoint, never a neighbour
    assert not eq[~keep].any() and np.array_equal(eq[keep], eigs)


def test_cpu_iss_matches_numpy_restatement(oracle):
    rng = np.random.default_rng(5)
    # 5000 points: three noisy planes and two blobs in a 400 mm box (keypoints where the planes meet and on the blobs)
    parts = []
    for k in range(3):
        P = rng.uniform(0.0, 400.0, (1200, 3))
        P[:, k] = 200.0 + rng.normal(0.0, 3.0, 1200)
        parts.append(P)
    parts += [rng.normal(c, 25.0, (700, 3)) for c in ((100.0, 100.0, 300.0), (300.0, 300.0, 100.0))]
    xyz = np.concatenate(parts)[:5000].astype(np.float32)
    assert len(xyz) == 5000
    for prm in (DEFAULTS, dict(DEFAULTS, salient_radius=120.0, non_max_radius=80.0)):
        kp, eigs = iss_oracle.iss(oracle.Cloud(xyz), **prm, want_eigs=True)
        kn, en = _numpy_iss(xyz, **prm)
        assert len(kn) >= 5
        _compare_eigs(eigs, en, "oracle vs numpy")
        _compare_keypoints(kp, kn, xyz, en, prm, "oracle vs numpy")


def test_cpu_kp_repeatability_known_answers(oracle):
    rng = np.random.default_rng(9)
    a = rng.uniform(-5000.0, 5000.0, (400, 3)).astype(np.float32)
    r = iss_oracle.kp_repeatability(a, a)
    assert r["rate"] == 1.0 and np.array_equal(r["nn_idx"], np.arange(400)) and not r["nn_dist"].any()
    for shift, hits in ((29.0, 400), (31.0, 0)):
        r = iss_oracle.kp_repeatability(a, a + np.float32([shift, 0, 0]), radius=30.0)
        assert r["hits"] == hits and np.array_equal(r["nn_idx"], np.arange(400))
    # a pose moves the sets: B = R A + t given as raw points, undone by pose_b = [R|t]^-1 ... applied to B
    yaw = np.deg2rad(20.0)
    R = np.array([[np.cos(yaw), -np.sin(yaw), 0], [np.sin(yaw), np.cos(yaw), 0], [0, 0, 1]])
    t = np.array([1500.0, -700.0, 40.0])
    b = (a.astype(np.float64) @ R.T + t).astype(np.float32)
    assert iss_oracle.kp_repeatability(a, b)["hits"] < 10
    pose_b = np.hstack([R.T, (-R.T @ t)[:, None]])
    r = iss_oracle.kp_repeatability(a, b, pose_b=pose_b)
    assert r["hits"] == 400 and np.array_equal(r["nn_idx"], np.arange(400))
    pose_a = np.hstack([R, t[:, None]])
    r = iss_oracle.kp_repeatability(a, b, pose_a=pose_a)
    assert r["hits"] == 400 and np.array_equal(r["nn_idx"], np.arange(400))
    r = iss_oracle.kp_repeatability(a, np.zeros((0, 3), np.float32))
    assert r["hits"] == 0 and (r["nn_idx"] == -1).all() and np.isinf(r["nn_dist"]).all()


# ---- GPU: bshot_detect_iss / bshot_kp_repeatability --------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("sensor", ["hdl32e", "hdl64e"])
@pytest.mark.parametrize("radii", [(60.0, 40.0), (200.0, 130.0), (1000.0, 600.0)])
def test_detect_iss_parity(bshot, oracle, synth, gpu_ctx, sensor, radii):
    xyz = synth.make_scan(sensor, 0)
    prm = dict(DEFAULTS, salient_radius=radii[0], non_max_radius=radii[1])
    gpu_ctx.set_cloud(xyz)
    g = gpu_ctx.detect_iss(bshot.iss_default_params(**prm), want_eigs=True)
    kp, eigs = iss_oracle.iss(oracle.Cloud(xyz), **prm, want_eigs=True)
    print(f"{sensor} r_s={radii[0]}: {len(g['idx'])} device / {len(kp)} oracle keypoints")
    assert len(kp) > 0
    _compare_eigs(g["eigs"], eigs, f"{sensor} {radii}")
    _compare_keypoints(g["idx"], kp, xyz, eigs, prm, f"{sensor} {radii}")
    assert np.all(np.diff(g["idx"]) > 0)
    assert np.array_equal(g["xyz"], xyz[g["idx"]])


@pytest.mark.gpu
def test_detect_iss_known_answers(bshot, oracle, gpu_ctx):
    prm = bshot.iss_default_params(**DEFAULTS)
    for seed in range(4):
        P = _corner(seed)
        gpu_ctx.set_cloud(P)
        assert np.array_equal(gpu_ctx.detect_iss(prm)["idx"], iss_oracle.iss(oracle.Cloud(P), **DEFAULTS))
    gpu_ctx.set_cloud(_plane(1))
    assert len(gpu_ctx.detect_iss(prm)["idx"]) == 0
    P = _plane(2, n=40, xy_noise=0.0, z_noise=1.0)
    gpu_ctx.set_cloud(P)
    assert np.array_equal(gpu_ctx.detect_iss(prm)["idx"], iss_oracle.iss(oracle.Cloud(P), **DEFAULTS))
    gpu_ctx.set_cloud(np.zeros((0, 3), np.float32))                    # empty cloud: count 0, status OK
    g = gpu_ctx.detect_iss(prm, want_eigs=True)
    assert len(g["idx"]) == 0 and g["eigs"].shape == (0, 3)
    gpu_ctx.set_cloud(_corner(0)[:4])
    g = gpu_ctx.detect_iss(prm, want_eigs=True)
    assert len(g["idx"]) == 0 and not g["eigs"].any()
    P = _corner(3)
    Q = np.insert(P, [0, 50, 200], np.array([[np.nan, 0, 0], [0, np.inf, 0], [1.0, 2.0, -np.inf]], np.float32), axis=0)
    gpu_ctx.set_cloud(Q)
    g = gpu_ctx.detect_iss(prm, want_eigs=True)
    kq, eq = iss_oracle.iss(oracle.Cloud(Q), **DEFAULTS, want_eigs=True)
    assert np.array_equal(g["idx"], kq)
    keep = np.isfinite(Q).all(1)
    assert not g["eigs"][~keep].any()
    _compare_eigs(g["eigs"], eq, "NaN points")


@pytest.mark.gpu
def test_detect_iss_capacity_and_arguments(bshot, synth):
    L = bshot.lib()
    import ctypes as C
    with bshot.Context(0, 131072, 1024, 1024) as ctx:
        prm = bshot.iss_default_params()
        cnt = C.c_size_t()
        assert L.bshot_detect_iss(ctx.h, C.byref(prm), None, None, 0, C.byref(cnt), None) == -4  # BSHOT_E_STATE: no cloud yet
        assert b"no cloud" in L.bshot_last_error()
        xyz = synth.make_scan("hdl64e", 0)
        ctx.set_cloud(xyz)
        full = ctx.detect_iss(prm)
        k = len(full["idx"])
        assert k > 20
        cap = k // 3
        idx = np.full(k, -7, np.int32)
        kxyz = np.zeros((k, 3), np.float32)
        rc = L.bshot_detect_iss(ctx.h, C.byref(prm), bshot._p(idx), bshot._p(kxyz), cap, C.byref(cnt), None)
        assert rc == bshot.E_CAPACITY and cnt.value == k
        assert np.array_equal(idx[:cap], full["idx"][:cap]) and (idx[cap:] == -7).all()
        assert np.array_equal(kxyz[:cap], full["xyz"][:cap])
        for bad in (dict(salient_radius=0.0), dict(non_max_radius=-1.0), dict(min_neighbors=0), dict(gamma_21=float("nan")),
                    dict(gamma_32=float("inf")), dict(salient_radius=float("nan"))):
            p = bshot.iss_default_params(**bad)
            assert L.bshot_detect_iss(ctx.h, C.byref(p), None, None, 0, C.byref(cnt), None) == -1, bad
        assert L.bshot_kp_repeatability(ctx.h, bshot._p(xyz), 10, None, bshot._p(xyz), 10, None, 0.0, None, None, None) == -1


def _frame_loop(bshot, synth, with_iss, process_frame=False):
    """four frames through the frame-to-map flow (or bshot_process_frame), optionally with an ISS call after the
    extraction; returns everything the loop produced"""
    p = bshot.default_params(top_k=600)
    out = []
    with bshot.Context(0, 131072, 1024, 1 << 15) as ctx:
        if process_frame:
            for k in range(4):
                f = ctx.process_frame(synth.make_scan("hdl32e", k), p)
                if with_iss:
                    ctx.detect_iss()
                out += [f["kp_idx"], f["bits"], f["pairs"]]
            return out
        ctx.gmap_create(1 << 15, 4096)
        pose = np.eye(4, dtype=np.float32)[:3].copy()
        for k in range(4):
            f = ctx.extract_frame(synth.make_scan("hdl32e", k), p)
            if with_iss:
                ctx.detect_iss()
            if k:
                r = ctx.match_frame_to_map(pose[:, 3], 100000.0, pose)
                out += [r["pairs"], r["target_xyz"]]
            pose[0, 3] = 500.0 * k
            ctx.gmap_update_from_frame(pose)
            ctx.frame_commit()
            out += [f["kp_idx"], f["bits"], f["kp_xyz"], f["seg_ratio"]]
        xyz, desc = ctx.gmap_get_keypoints(np.zeros(3, np.float32), 100000.0)
        out += [xyz, desc]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("process_frame", [False, True])
def test_detect_iss_has_no_side_effects(bshot, synth, process_frame):
    a = _frame_loop(bshot, synth, False, process_frame)
    b = _frame_loop(bshot, synth, True, process_frame)
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8))


@pytest.mark.gpu
def test_iss_keypoints_through_bshot(bshot, oracle, synth, gpu_ctx):
    xyz = synth.make_scan("hdl64e", 0)
    gpu_ctx.set_cloud(xyz)
    g = gpu_ctx.detect_iss()
    assert len(g["idx"]) > 100
    gpu_ctx.set_keypoints(g["xyz"])
    bits = gpu_ctx.compute_descriptors(bshot.default_params())
    od = oracle.Cloud(xyz).compute_descriptors(g["xyz"], 3000.0, 300, oracle.MODE_REFERENCE)
    same = (synth.unpack_bits(bits) == synth.unpack_bits(od["bits"])).mean()
    assert same >= 0.999, same


def _frame_pose(k):
    yaw = np.deg2rad(0.5 * k)
    T = np.eye(4, dtype=np.float32)[:3]
    T[:2, :2] = [[np.cos(yaw), -np.sin(yaw)], [np.sin(yaw), np.cos(yaw)]]
    T[0, 3] = 500.0 * k
    return T


@pytest.mark.gpu
def test_kp_repeatability_matches_oracle(bshot, oracle, synth, gpu_ctx):
    kps = []
    for k in (0, 1):
        gpu_ctx.set_cloud(synth.make_scan("hdl32e", k))
        kps.append(gpu_ctx.detect_iss(bshot.iss_default_params(salient_radius=200.0, non_max_radius=130.0))["xyz"])
    for pa, pb in ((None, None), (_frame_pose(1), _frame_pose(0)), (_frame_pose(0), _frame_pose(1))):
        g = gpu_ctx.kp_repeatability(kps[1], kps[0], pa, pb, 30.0)
        o = iss_oracle.kp_repeatability(kps[1], kps[0], pa, pb, 30.0)
        assert np.array_equal(g["nn_idx"], o["nn_idx"]) and g["hits"] == o["hits"]
        assert np.array_equal(g["nn_dist"].view(np.uint32), o["nn_dist"].view(np.uint32))
    r = gpu_ctx.kp_repeatability(kps[1], kps[0], _frame_pose(1), _frame_pose(0), 30.0)
    print(f"ISS repeat rate frame 1 -> 0 (r_s 200): {r['rate']:.3f} of {len(kps[1])}")
    assert r["hits"] > 0
    a = kps[0]
    for shift, hits in ((29.0, len(a)), (31.0, 0)):
        assert gpu_ctx.kp_repeatability(a, a + np.float32([0, 0, shift]))["hits"] == hits
    e = gpu_ctx.kp_repeatability(a, np.zeros((0, 3), np.float32))
    assert e["hits"] == 0 and (e["nn_idx"] == -1).all()


@pytest.fixture(scope="module")
def iss_shim_binary(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("iss_shim") / "host_shim_iss_test")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror",
                           os.path.join(ROOT, "tests", "host_shim_iss_test.cpp"), "-o", out, "-L", PKG, "-lbshot_b200",
                           f"-Wl,-rpath,{PKG}"])
    return out


def test_iss_shim_compiles(iss_shim_binary):
    assert os.path.exists(iss_shim_binary)


@pytest.mark.gpu
def test_iss_shim_kp_evaluation(iss_shim_binary, bshot, synth, tmp_path):
    """setSrcFrame -> extractKeypoints -> issKpDetection -> computeDescriptors -> featureMatching -> evaluateEstimation ->
    poseEstimation -> updateMap -> kpEvaluation over two frames; the repeat rates equal the Python path's on the same
    keypoints and poses"""
    scans = [synth.make_scan("hdl32e", f)[::2].copy() for f in (0, 1)]
    paths = []
    for i, s in enumerate(scans):
        paths.append(str(tmp_path / f"cloud{i}.bin"))
        s.tofile(paths[-1])
    outp = str(tmp_path / "out.bin")
    r = subprocess.run([iss_shim_binary, paths[0], paths[1], outp], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = open(outp, "rb").read()
    off, frames = 0, []
    for _ in range(2):
        nk, ni = struct.unpack_from("ii", raw, off); off += 8
        kp = np.frombuffer(raw, np.float32, 3 * nk, off).reshape(nk, 3); off += 12 * nk
        iss = np.frombuffer(raw, np.float32, 3 * ni, off).reshape(ni, 3); off += 12 * ni
        pose = np.frombuffer(raw, np.float32, 16, off).reshape(4, 4); off += 64
        sr_rate, iss_rate = struct.unpack_from("dd", raw, off); off += 16
        frames.append((kp, iss, pose, sr_rate, iss_rate))
    assert off == len(raw)
    with bshot.Context(0, 131072, 1024, 1024) as ctx:
        for k in range(2):
            ctx.set_cloud(scans[k])
            assert np.array_equal(ctx.detect_iss()["xyz"], frames[k][1])
        # frame 0 is its own reference frame (src/lidar_odometry.cpp:187-194): both rates are 1
        for k, ref in ((0, 0), (1, 0)):
            kp, iss, pose, sr_rate, iss_rate = frames[k]
            assert len(iss) > 0
            want_sr = ctx.kp_repeatability(kp, frames[ref][0], pose, frames[ref][2], 30.0)["rate"]
            want_iss = ctx.kp_repeatability(iss, frames[ref][1], pose, frames[ref][2], 30.0)["rate"]
            print(f"host shim frame {k}: repeat rates seg-ratio {sr_rate:.4f}, ISS {iss_rate:.4f}")
            assert sr_rate == want_sr and iss_rate == want_iss
        assert frames[0][3] == 1.0 and frames[0][4] == 1.0
