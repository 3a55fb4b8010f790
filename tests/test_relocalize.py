"""Saving, restoring and relocalising in the GPU-resident map: bshot_gmap_export (the whole map in map order),
bshot_gmap_import (the map rebuilt exactly, without the admission rule) and bshot_relocalize / _cloud (a scan against
every map entry: mutual nearest neighbours -> RANSAC -> ICP around T_ransac -> the step's tail when accepted).

The front end carries the reference's persistent normals from one extraction to the next, so a twin context that must
give the same descriptors replays the same extractions (extract_scan) instead of the calls under test."""
import ctypes
import functools
import os
import subprocess

import numpy as np
import pytest

from test_odometry_step import assert_same_report, chain_step

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "b-shot-slam_b200")

MAP_ENTRIES, MAP_BLOCKS = 1 << 16, 4096


# ---- helpers ----------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def lasers(synth, k):
    return synth.make_lasers("hdl32e", k)


def step(ctx, L, p):
    return ctx.odometry_step(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p)


def extract(ctx, L, p):
    return ctx.extract_scan(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p.front, vert_init=p.vert_init_rad, lowpt_th=p.lowpt_th,
                            want_cloud=False)


def relocalize(ctx, L, p, min_inliers=15):
    return ctx.relocalize(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p, min_inliers=min_inliers)


def mapped(bshot, synth, frames, p, max_targets=1 << 16):
    """a context whose map holds the odometry of these rotations"""
    ctx = bshot.Context(0, 131072, 1024, max_targets)
    ctx.gmap_create(MAP_ENTRIES, MAP_BLOCKS)
    for k in frames:
        step(ctx, lasers(synth, k), p)
    return ctx


def fresh(bshot, max_targets=1 << 16, max_entries=MAP_ENTRIES):
    ctx = bshot.Context(0, 131072, 1024, max_targets)
    ctx.gmap_create(max_entries, MAP_BLOCKS)
    return ctx


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32 if a.dtype == np.float32 else a.dtype), b.view(np.uint32 if b.dtype == np.float32 else b.dtype))


def block_coords(xyz):
    """roundf(p / 10 m) per axis (half away from zero), as the map computes a block's lattice coordinates"""
    q = (np.asarray(xyz, np.float32) / np.float32(10000.0)).astype(np.float64)
    return (np.sign(q) * np.floor(np.abs(q) + 0.5)).astype(np.int64)


def mul4x4(a, b):
    """odom_math.cuh's mul4x4 in fp32: ((a0 b0 + a1 b1) + a2 b2) + a3 b3"""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    o = np.empty((4, 4), np.float32)
    for i in range(4):
        for j in range(4):
            o[i, j] = ((a[i, 0] * b[0, j] + a[i, 1] * b[1, j]) + a[i, 2] * b[2, j]) + a[i, 3] * b[3, j]
    return o


def host_relocalize(ctx, L, p, xyzr, desc, min_inliers=15):
    """the relocalisation as a composition of host calls on a context holding the same map: extract_scan, match_mutual
    against the exported map, ransac, gmap_get_keypoints around T_ransac, icp, mul4x4"""
    f = extract(ctx, L, p)
    pairs = ctx.match_mutual(f["bits"], desc)[0] if len(desc) else np.empty((0, 2), np.int32)
    rs = ctx.ransac(f["kp_xyz"], xyzr[:, :3], pairs, p.ransac_iterations, p.inlier_threshold)
    T_r = rs["transform"]
    n_icp, icp_it, T_best = 0, 0, T_r
    if p.run_icp:
        tx, _ = ctx.gmap_get_keypoints(T_r[:3, 3], p.map_range)
        ic = ctx.icp(f["kp_xyz"], tx, pre=T_r, max_iterations=10)
        n_icp, icp_it, T_best = len(tx), ic["iterations"], mul4x4(ic["transform"], T_r)
    n_inl = len(rs["pairs"])
    return dict(pose=T_best, T_ransac=T_r, n_points=f["n_points"], n_map=len(desc), n_icp_targets=n_icp, n_keypoints=len(f["bits"]),
                n_pairs=len(pairs), n_inliers=n_inl, ransac_iterations=rs["iterations"], icp_iterations=icp_it, accepted=int(n_inl >= min_inliers))


def assert_same_reloc(dev, host, where=""):
    for key in ("pose", "T_ransac"):
        assert same_bits(np.asarray(dev[key], np.float32), np.asarray(host[key], np.float32)), (where, key, dev[key], host[key])
    for key in ("n_points", "n_map", "n_icp_targets", "n_keypoints", "n_pairs", "n_inliers", "ransac_iterations", "icp_iterations", "accepted"):
        assert int(dev[key]) == int(host[key]), (where, key, dev[key], host[key])


def pose_error(T, R_true, t_true):
    """translation error (mm) and rotation error (deg) of a 4 x 4 pose"""
    T = np.asarray(T, np.float64)
    dt = float(np.linalg.norm(T[:3, 3] - np.asarray(t_true, np.float64)))
    c = (np.trace(T[:3, :3] @ np.asarray(R_true, np.float64).T) - 1.0) / 2.0
    return dt, float(np.degrees(np.arccos(np.clip(c, -1.0, 1.0))))


def rot_z(deg):
    a = np.radians(deg)
    return np.array([[np.cos(a), -np.sin(a), 0.0], [np.sin(a), np.cos(a), 0.0], [0.0, 0.0, 1.0]])


def distractors(synth, n, seed=11):
    """n entries with random <= 40-bit descriptors in blocks 1 km and more from the route (beyond any map_range used)"""
    rng = np.random.default_rng(seed)
    xyzr = np.empty((n, 4), np.float32)
    xyzr[:, 0] = np.round(rng.uniform(1.0e6, 1.6e6, n) / 10.0) * 10.0
    xyzr[:, 1] = np.round(rng.uniform(-3.0e5, 3.0e5, n) / 10.0) * 10.0
    xyzr[:, 2] = np.round(rng.uniform(-5.0e3, 5.0e3, n) / 10.0) * 10.0
    xyzr[:, 3] = rng.uniform(0.0, 1.0, n).astype(np.float32)
    return xyzr, synth.random_descriptors(n, seed=seed, density=40)


# ---- CPU --------------------------------------------------------------------------------------------------------------------
def test_reloc_symbols_exported(bshot):
    L = bshot.lib()
    for s in ("bshot_gmap_export", "bshot_gmap_import", "bshot_relocalize", "bshot_relocalize_cloud"):
        assert s in bshot.EXPORTS and hasattr(L, s), s
    assert bshot.RelocReport.pose.offset == 0 and bshot.RelocReport.n_points.offset == 128
    assert bshot.RelocReport.n_keypoints.offset == 152 and ctypes.sizeof(bshot.RelocReport) == 176


def test_block_coords_round_half_away():
    assert list(block_coords([5000.0, -5000.0, 4990.0])) == [1, -1, 0]
    assert list(block_coords([15000.0, -14990.0, 0.0])) == [2, -1, 0]


@pytest.fixture(scope="module")
def reloc_shim_binary(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("reloc_shim") / "host_shim_relocalize_test")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror",
                           os.path.join(ROOT, "tests", "host_shim_relocalize_test.cpp"), "-o", out, "-L", PKG, "-lbshot_b200",
                           f"-Wl,-rpath,{PKG}"])
    return out


def _write_rotations(tmp_path, synth, frames):
    L0 = synth.make_lasers("hdl32e", frames[0])
    ring = str(tmp_path / "ring.bin")
    np.ascontiguousarray(L0["ring_deg"], np.float64).tofile(ring)
    rec = np.dtype([("az", "<f8"), ("ve", "<f8"), ("di", "<u2")])
    paths = {}
    for f in frames:
        L = synth.make_lasers("hdl32e", f)
        a = np.empty(len(L["azimuth"]), rec)
        a["az"], a["ve"], a["di"] = L["azimuth"], L["vertical"], L["distance"]
        paths[f] = str(tmp_path / f"rot{f}.bin")
        a.tofile(paths[f])
    return ring, paths


def test_relocalize_shim_fails_loudly_without_gpu(reloc_shim_binary, tmp_path, synth):
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    ring, paths = _write_rotations(tmp_path, synth, [0, 1])
    r = subprocess.run([reloc_shim_binary, ring, str(tmp_path / "out.bin"), paths[1], paths[1], paths[0]], capture_output=True, text=True)
    assert r.returncode == 1 and "no CUDA device" in r.stdout


# ---- GPU: export and import -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_export_is_map_order(bshot, synth):
    """export = getKeypoints over a cube covering every block, bit for bit; two runs of the same steps export the same
    arrays whatever order the admission kernel gave the pool"""
    p = bshot.odom_default_params(top_k=600)
    with mapped(bshot, synth, range(12), p) as a, mapped(bshot, synth, range(12), p) as b:
        xa, da = a.gmap_export()
        xb, db = b.gmap_export()
        assert len(xa) == a.gmap_size()[0] > 0
        assert same_bits(xa, xb) and np.array_equal(da, db)
        lo, hi = xa[:, :3].min(axis=0), xa[:, :3].max(axis=0)
        centre = ((lo + hi) / 2.0).astype(np.float32)
        rng = float(np.max(hi - lo) / 2.0 + 10000.0)
        x, d = a.gmap_get_keypoints(centre, rng)
        assert same_bits(xa[:, :3].copy(), x) and np.array_equal(da, d)
        # map order: blocks ascending in (x, y, z), one run per block
        bc = block_coords(xa[:, :3])
        keys = (bc[:, 0] + (1 << 20)) * (1 << 42) + (bc[:, 1] + (1 << 20)) * (1 << 21) + (bc[:, 2] + (1 << 20))
        assert np.all(np.diff(keys) >= 0)


@pytest.mark.gpu
def test_import_round_trip(bshot, synth):
    """export A -> import B -> export B is the identity; relocalisation and steps after the import give A's reports and
    A's final map bit for bit (admission and overwrite against imported entries); an order that keeps each block's
    relative order imports to the same map"""
    p = bshot.odom_default_params(top_k=600)
    with mapped(bshot, synth, range(8), p) as a, fresh(bshot) as b:
        for k in range(8):   # the same front-end history as A (persistent normals)
            extract(b, lasers(synth, k), p)
        xa, da = a.gmap_export()
        b.gmap_import(xa, da)
        xb, db = b.gmap_export()
        assert same_bits(xa, xb) and np.array_equal(da, db)
        assert a.gmap_size() == b.gmap_size()
        ra, rb = relocalize(a, lasers(synth, 8), p), relocalize(b, lasers(synth, 8), p)
        assert_same_reloc(rb, ra, "reloc")
        assert ra["accepted"] == 1
        for k in (9, 10, 11):
            assert_same_report(step(b, lasers(synth, k), p), step(a, lasers(synth, k), p), k)
            assert a.gmap_size() == b.gmap_size(), k
        xa2, da2 = a.gmap_export()
        xb2, db2 = b.gmap_export()
        assert len(xa2) > len(xa)
        assert same_bits(xa2, xb2) and np.array_equal(da2, db2)

        # a shuffle that keeps each block's relative order
        bc = block_coords(xa2[:, :3])
        _, blk = np.unique(bc, axis=0, return_inverse=True)
        blk = blk.reshape(-1)
        perm = np.random.default_rng(5).permutation(len(xa2))
        order = np.empty(len(xa2), np.int64)
        for bid in np.unique(blk):
            slots = np.flatnonzero(blk[perm] == bid)
            order[slots] = np.flatnonzero(blk == bid)
        assert not np.array_equal(order, np.arange(len(order)))
        b.gmap_import(xa2[order], da2[order])
        xs, ds = b.gmap_export()
        assert same_bits(xs, xa2) and np.array_equal(ds, da2)


@pytest.mark.gpu
def test_import_errors(bshot, synth):
    p = bshot.odom_default_params(top_k=600)
    with mapped(bshot, synth, range(3), p) as a, fresh(bshot, max_entries=256) as b:
        x, d = a.gmap_export()
        assert 256 < len(x)
        bad = x[:100].copy()
        bad[17, 1] = np.nan
        b.gmap_import(x[:100], d[:100])
        with pytest.raises(bshot.BshotError) as e:
            b.gmap_import(bad, d[:100])
        assert e.value.code == bshot.E_INVALID
        assert b.gmap_size() == (0, 0) and len(b.gmap_export()[0]) == 0
        bad[17, 1] = np.inf
        with pytest.raises(bshot.BshotError) as e:
            b.gmap_import(bad, d[:100])
        assert e.value.code == bshot.E_INVALID
        b.gmap_import(x[:100], d[:100])
        with pytest.raises(bshot.BshotError) as e:
            b.gmap_import(x, d)   # more than max_entries
        assert e.value.code == bshot.E_CAPACITY
        assert b.gmap_size() == (0, 0)
        b.gmap_import(x[:100], d[:100])
        assert b.gmap_size()[0] == 100
        b.gmap_import(x[:0], d[:0])
        assert b.gmap_size() == (0, 0) and len(b.gmap_export()[0]) == 0
        # more blocks than the table holds: every entry in a block of its own
        many = np.zeros((3000, 4), np.float32)
        many[:, 0] = np.arange(3000, dtype=np.float32) * 20000.0
        c = bshot.Context(0, 131072, 1024, 1 << 16)
        try:
            c.gmap_create(4096, 64)
            with pytest.raises(bshot.BshotError) as e:
                c.gmap_import(many, np.zeros((3000, 6), np.uint64))
            assert e.value.code == bshot.E_CAPACITY
            assert c.gmap_size() == (0, 0)
        finally:
            c.close()
    with bshot.Context(0, 131072, 1024, 1 << 16) as c:
        for call in (lambda: c.gmap_export(), lambda: c.gmap_import(x[:1], d[:1])):
            with pytest.raises(bshot.BshotError) as e:
                call()
            assert e.value.code == bshot.E_STATE


# ---- GPU: relocalisation -------------------------------------------------------------------------------------------------
def _reloc_vs_host(bshot, synth, xyzr, desc, p, queries, matcher=-1, min_nm_pairs=None):
    """device relocalisation vs the host composition on two contexts holding the same imported map; when accepted, the
    next two scans by odometry_step against the five-call chain"""
    with fresh(bshot, max_targets=1 << 17) as dev, fresh(bshot, max_targets=1 << 17) as host:
        for c in (dev, host):
            c.set_matcher(matcher)
            c.gmap_import(xyzr, desc)
        if min_nm_pairs is not None:
            assert 600 * len(desc) >= min_nm_pairs, len(desc)
        accepted = 0
        for q in queries:
            rd = relocalize(dev, lasers(synth, q), p)
            rh = host_relocalize(host, lasers(synth, q), p, xyzr, desc)
            assert_same_reloc(rd, rh, q)
            if not rd["accepted"]:
                continue
            accepted += 1
            host.gmap_update_from_frame(rh["pose"][:3])
            host.frame_commit()
            state = dict(pose_ref=rh["pose"], initial=False)
            for k in (q + 1, q + 2):
                assert_same_report(step(dev, lasers(synth, k), p), chain_step(host, state, p, lasers=lasers(synth, k)), (q, k))
            xd, dd = dev.gmap_export()
            xh, dh = host.gmap_export()
            assert same_bits(xd, xh) and np.array_equal(dd, dh)
            # the next query starts from the imported map again
            for c in (dev, host):
                c.odometry_reset()
                c.gmap_import(xyzr, desc)
        return accepted


@pytest.mark.gpu
@pytest.mark.parametrize("run_icp", [1, 0])
def test_relocalize_equals_host_small_map(bshot, synth, run_icp):
    """4 mapped rotations: fewer than 2^21 pairs, the XOR + POPC matcher by size"""
    p = bshot.odom_default_params(top_k=600, run_icp=run_icp)
    with mapped(bshot, synth, range(4), p) as a:
        x, d = a.gmap_export()
    assert 600 * len(d) < (1 << 21)
    assert _reloc_vs_host(bshot, synth, x, d, p, [2, 5]) >= 1


@pytest.mark.gpu
@pytest.mark.parametrize("matcher", [-1, 0])
def test_relocalize_equals_host_tensor_core_map(bshot, synth, matcher):
    """12 mapped rotations plus 8000 distant distractors: above 2^21 pairs, so AUTO takes the tensor-core pipeline;
    the same forced onto XOR + POPC"""
    p = bshot.odom_default_params(top_k=600)
    with mapped(bshot, synth, range(12), p) as a:
        x, d = a.gmap_export()
    dx, dd = distractors(synth, 8000)
    xyzr, desc = np.concatenate([x, dx]), np.concatenate([d, dd])
    assert _reloc_vs_host(bshot, synth, xyzr, desc, p, [3, 9], matcher=matcher, min_nm_pairs=1 << 21) >= 1


@pytest.mark.gpu
def test_relocalize_recovers_ground_truth(bshot, synth):
    """a mapped rotation and a scan at an unmapped pose with a yaw far from the route's, against a restored map.
    Ground truth in the map frame (rotation 0's sensor frame): rotation k at (500 k, 0, 0) without yaw; the scan below
    at (2750, 0, 0) yawed by 40 degrees.
    Measured on one NVIDIA B200: rotation 6 47.1 mm / 0.21 deg, the step to rotation 7 67.2 mm / 0.13 deg, the unmapped
    pose 46.3 mm / 0.26 deg; the tolerances leave a margin of about 4x."""
    TOL_MM, TOL_DEG = 300.0, 1.0
    p = bshot.odom_default_params(top_k=600)
    with mapped(bshot, synth, range(12), p) as a:
        x, d = a.gmap_export()
    with fresh(bshot) as b:
        b.gmap_import(x, d)
        j = 6
        r = relocalize(b, lasers(synth, j), p)
        dt, da = pose_error(r["pose"], np.eye(3), [500.0 * j, 0.0, 0.0])
        print(f"mapped rotation {j}: accepted {r['accepted']}, {r['n_inliers']} inliers, error {dt:.1f} mm {da:.3f} deg")
        assert r["accepted"] == 1 and dt < TOL_MM and da < TOL_DEG, (dt, da, r)
        s = step(b, lasers(synth, j + 1), p)
        dt, da = pose_error(s["pose"], np.eye(3), [500.0 * (j + 1), 0.0, 0.0])
        print(f"step to rotation {j + 1}: {s['n_inliers']} inliers, update {s['should_update_map']}, error {dt:.1f} mm {da:.3f} deg")
        assert s["was_initial"] == 0 and dt < TOL_MM and da < TOL_DEG, (dt, da, s)
    with fresh(bshot) as b:
        b.gmap_import(x, d)
        yaw = 40.0
        cloud = synth.make_scan("hdl32e", 0, pos=[2750.0, 0.0, 550.0], yaw_deg=yaw)
        # the map was built from preprocessed rotations, which hold nothing below the low-point threshold; the same cut
        # here (without it the object bases below it pull ICP about 2 m up)
        cloud = cloud[cloud[:, 2] >= p.lowpt_th]
        r = b.relocalize_cloud(cloud, p)
        dt, da = pose_error(r["pose"], rot_z(yaw), [2750.0, 0.0, 0.0])
        print(f"novel pose: accepted {r['accepted']}, {r['n_inliers']} inliers of {r['n_pairs']} pairs, error {dt:.1f} mm {da:.3f} deg")
        assert r["accepted"] == 1 and dt < TOL_MM and da < TOL_DEG, (dt, da, r)


@pytest.mark.gpu
def test_rejection_leaves_state(bshot, synth):
    """an empty map and min_inliers above K: accepted = 0, and the next step equals that of a twin that only extracted"""
    p = bshot.odom_default_params(top_k=600)
    with fresh(bshot) as a, fresh(bshot) as t:
        r = relocalize(a, lasers(synth, 0), p)
        assert r["accepted"] == 0 and r["n_map"] == 0 and r["n_pairs"] == 0
        extract(t, lasers(synth, 0), p)
        for k in (1, 2):
            assert_same_report(step(a, lasers(synth, k), p), step(t, lasers(synth, k), p), k)
        assert a.gmap_size() == t.gmap_size()
    with mapped(bshot, synth, range(4), p) as a, mapped(bshot, synth, range(4), p) as t:
        size = a.gmap_size()
        r = relocalize(a, lasers(synth, 4), p, min_inliers=10 ** 6)
        assert r["accepted"] == 0 and r["n_inliers"] >= 15 and a.gmap_size() == size
        extract(t, lasers(synth, 4), p)
        for k in (5, 6):
            assert_same_report(step(a, lasers(synth, k), p), step(t, lasers(synth, k), p), k)
        xa, da = a.gmap_export()
        xt, dt = t.gmap_export()
        assert same_bits(xa, xt) and np.array_equal(da, dt)
        for bad in (2, 0, -1):
            with pytest.raises(bshot.BshotError) as e:
                relocalize(a, lasers(synth, 7), p, min_inliers=bad)
            assert e.value.code == bshot.E_INVALID
    with bshot.Context(0, 131072, 1024, 1 << 16) as c:
        with pytest.raises(bshot.BshotError) as e:
            relocalize(c, lasers(synth, 0), p)
        assert e.value.code == bshot.E_STATE


@pytest.mark.gpu
def test_relocalize_icp_target_overflow_leaves_state(bshot, synth):
    """an ICP target set above max_targets: BSHOT_E_CAPACITY, and pose, status, map and reference frame unchanged"""
    p = bshot.odom_default_params(top_k=600)
    with mapped(bshot, synth, range(12), p) as a:
        x, d = a.gmap_export()
    with fresh(bshot, max_targets=1024) as c, fresh(bshot, max_targets=1024) as t:
        for ctx in (c, t):
            ctx.gmap_import(x, d)
        with pytest.raises(bshot.BshotError) as e:
            relocalize(c, lasers(synth, 6), p)
        assert e.value.code == bshot.E_CAPACITY
        extract(t, lasers(synth, 6), p)
        assert c.gmap_size() == t.gmap_size()
        s_c, s_t = step(c, lasers(synth, 7), bshot.odom_default_params(top_k=600, map_range=5000.0)), \
            step(t, lasers(synth, 7), bshot.odom_default_params(top_k=600, map_range=5000.0))
        assert s_c["was_initial"] == 1
        assert_same_report(s_c, s_t)


@pytest.mark.gpu
def test_device_odometry_relocalize_shim_equals_python(bshot, synth, reloc_shim_binary, tmp_path):
    ring, paths = _write_rotations(tmp_path, synth, [0, 1, 2, 3, 4, 5, 6])
    out = str(tmp_path / "out.bin")
    r = subprocess.run([reloc_shim_binary, ring, out, paths[5], paths[6]] + [paths[k] for k in range(5)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = np.fromfile(out, np.uint8)
    assert raw.size == 64 + 20 + 64
    p = bshot.odom_default_params()
    with mapped(bshot, synth, range(5), p) as a, fresh(bshot) as b:
        x, d = a.gmap_export()
        b.gmap_import(x, d)
        rl = relocalize(b, lasers(synth, 5), p)
        s = step(b, lasers(synth, 6), p)
    fields = raw[64:84].view(np.int32)
    assert same_bits(raw[:64].view(np.float32).reshape(4, 4), rl["pose"])
    assert list(fields) == [len(d), rl["n_keypoints"], rl["n_pairs"], rl["n_inliers"], rl["accepted"]]
    assert same_bits(raw[84:].view(np.float32).reshape(4, 4), s["pose"])
