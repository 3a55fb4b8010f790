"""The per-scan odometry step (bshot_odometry_step / _cloud, bshot_ransac_dev) against the five-call chain it replaces
(extract -> match_mutual / match_frame_to_map -> ransac -> evaluate_estimation -> gmap_update_from_frame + frame_commit):
every report field and the map must agree bit for bit (h_diff_rad within 2 ulp: device acosf)."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "b-shot-slam_b200")


# ---- fixtures / helpers -------------------------------------------------------------------------------------------------
def chain_step(ctx, state, p, lasers=None, cloud=None):
    """the five calls of tests/test_odometry_loop.py for one scan; state = dict(pose_ref, initial)"""
    if lasers is not None:
        L = lasers
        f = ctx.extract_scan(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p.front, vert_init=p.vert_init_rad, lowpt_th=p.lowpt_th,
                             want_cloud=False)
        n_points = f["n_points"]
    else:
        f = ctx.extract_frame(cloud, p.front)
        n_points = len(cloud)
    pose_ref = state["pose_ref"]
    if state["initial"]:
        pairs, tgt = ctx.match_mutual(f["bits"], f["bits"])[0], f["kp_xyz"]
        n_targets = len(tgt)
    else:
        r = ctx.match_frame_to_map(pose_ref[:3, 3], p.map_range, pose_ref[:3], target_cap=1 << 17)
        pairs, tgt, n_targets = r["pairs"], r["target_xyz"], r["n_targets"]
    rs = ctx.ransac(f["kp_xyz"], tgt, pairs, p.ransac_iterations, p.inlier_threshold)
    ev = ctx.evaluate_estimation(rs["transform"], pose_ref, len(rs["pairs"]), f["kp_xyz"], tgt, run_icp=bool(p.run_icp))
    ctx.gmap_update_from_frame(ev["T_best"][:3])
    ctx.frame_commit()
    ctx.sync()
    out = dict(pose=ev["T_best"], T_ransac=rs["transform"], n_points=n_points, n_targets=n_targets, n_keypoints=len(f["bits"]),
               n_pairs=len(pairs), n_inliers=len(rs["pairs"]), ransac_iterations=rs["iterations"], icp_iterations=ev["icp_iterations"],
               should_update_map=int(ev["should_update_map"]), was_initial=int(state["initial"]), h_diff_rad=ev["h_diff"],
               t_diff_mm=ev["t_diff"])
    state["pose_ref"], state["initial"] = ev["T_best"], False
    return out


def assert_same_report(step, chain, where=""):
    for key in ("pose", "T_ransac"):
        assert np.array_equal(np.asarray(step[key], np.float32).view(np.uint32), np.asarray(chain[key], np.float32).view(np.uint32)), (where, key)
    for key in ("n_points", "n_targets", "n_keypoints", "n_pairs", "n_inliers", "ransac_iterations", "icp_iterations", "should_update_map",
                "was_initial"):
        assert int(step[key]) == int(chain[key]), (where, key, step[key], chain[key])
    assert np.float32(step["t_diff_mm"]).view(np.uint32) == np.float32(chain["t_diff_mm"]).view(np.uint32), where
    a, b = np.float32(step["h_diff_rad"]), np.float32(chain["h_diff_rad"])
    assert abs(int(a.view(np.int32)) - int(b.view(np.int32))) <= 2, (where, a, b)


def run_pair(bshot, inputs, p, kind, max_points=131072, max_kp=1024, max_targets=1 << 16):
    """the chain on context A and the step on context B over the same inputs, compared after every scan"""
    with bshot.Context(0, max_points, max_kp, max_targets) as a, bshot.Context(0, max_points, max_kp, max_targets) as b:
        a.gmap_create(1 << 16, 4096)
        b.gmap_create(1 << 16, 4096)
        state = dict(pose_ref=np.eye(4, dtype=np.float32), initial=True)
        reports = []
        for i, x in enumerate(inputs):
            if kind == "lasers":
                c = chain_step(a, state, p, lasers=x)
                s = b.odometry_step(x["azimuth"], x["vertical"], x["distance"], x["ring_deg"], p)
            else:
                c = chain_step(a, state, p, cloud=x)
                s = b.odometry_step_cloud(x, p)
            assert_same_report(s, c, i)
            assert a.gmap_size() == b.gmap_size(), i
            reports.append(s)
        pos = state["pose_ref"][:3, 3]
        xa, da = a.gmap_get_keypoints(pos, 100000.0)
        xb, db = b.gmap_get_keypoints(pos, 100000.0)
        assert np.array_equal(xa.view(np.uint32), xb.view(np.uint32)) and np.array_equal(da, db)
    return reports


# ---- CPU -----------------------------------------------------------------------------------------------------------------
def test_odom_params_default(bshot):
    p = bshot.odom_default_params()
    d = bshot.default_params()
    for name, _ in bshot.Params._fields_:
        assert getattr(p.front, name) == getattr(d, name), name
    assert p.vert_init_rad == -0.6 and p.lowpt_th == -1950.0 and p.map_range == 100000.0
    assert p.ransac_iterations == 2000 and p.inlier_threshold == 1500.0 and p.run_icp == 1
    q = bshot.odom_default_params(top_k=2048, run_icp=0)
    assert q.front.top_k == 2048 and q.run_icp == 0
    with pytest.raises(AttributeError):
        bshot.odom_default_params(no_such_field=1)


def test_odometry_symbols_exported(bshot):
    L = bshot.lib()
    for s in ("bshot_odom_params_default", "bshot_odometry_step", "bshot_odometry_step_cloud", "bshot_odometry_reset", "bshot_ransac_dev"):
        assert s in bshot.EXPORTS and hasattr(L, s), s


@pytest.fixture(scope="module")
def odometry_shim_binary(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("odometry_shim") / "host_shim_odometry_test")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror",
                           os.path.join(ROOT, "tests", "host_shim_odometry_test.cpp"), "-o", out, "-L", PKG, "-lbshot_b200",
                           f"-Wl,-rpath,{PKG}"])
    return out


def _write_rotations(tmp_path, synth, frames):
    L0 = synth.make_lasers("hdl32e", frames[0])
    ring = str(tmp_path / "ring.bin")
    np.ascontiguousarray(L0["ring_deg"], np.float64).tofile(ring)
    rec = np.dtype([("az", "<f8"), ("ve", "<f8"), ("di", "<u2")])
    paths, lasers = [], []
    for f in frames:
        L = synth.make_lasers("hdl32e", f)
        a = np.empty(len(L["azimuth"]), rec)
        a["az"], a["ve"], a["di"] = L["azimuth"], L["vertical"], L["distance"]
        path = str(tmp_path / f"rot{f}.bin")
        a.tofile(path)
        paths.append(path)
        lasers.append(L)
    return ring, paths, lasers


def test_device_odometry_shim_fails_loudly_without_gpu(odometry_shim_binary, tmp_path, synth):
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    ring, paths, _ = _write_rotations(tmp_path, synth, [0])
    r = subprocess.run([odometry_shim_binary, ring, str(tmp_path / "out.bin")] + paths, capture_output=True, text=True)
    assert r.returncode == 1 and "no CUDA device" in r.stdout


# ---- GPU: the step against the chain ----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_step_equals_chain_hdl32e(bshot, synth):
    p = bshot.odom_default_params(top_k=600)
    reps = run_pair(bshot, [synth.make_lasers("hdl32e", k) for k in range(12)], p, "lasers")
    assert reps[0]["was_initial"] == 1 and all(r["was_initial"] == 0 for r in reps[1:])
    for k, r in enumerate(reps):   # the sensor moves 500 mm a frame along x
        assert abs(r["pose"][0, 3] - 500.0 * k) < 350.0, (k, r["pose"])


@pytest.mark.gpu
def test_step_equals_chain_hdl64e(bshot, synth):
    p = bshot.odom_default_params(top_k=2048)
    run_pair(bshot, [synth.make_lasers("hdl64e", k) for k in range(4)], p, "lasers", max_points=1 << 18, max_kp=4096, max_targets=1 << 17)


@pytest.mark.gpu
def test_step_cloud_equals_chain(bshot, synth):
    p = bshot.odom_default_params(top_k=2048)
    run_pair(bshot, [synth.make_scan("hdl64e", k) for k in range(4)], p, "cloud", max_points=1 << 18, max_kp=4096, max_targets=1 << 17)


@pytest.mark.gpu
def test_step_equals_chain_without_icp(bshot, synth):
    p = bshot.odom_default_params(top_k=600, run_icp=0)
    reps = run_pair(bshot, [synth.make_lasers("hdl32e", k) for k in range(5)], p, "lasers")
    assert all(r["icp_iterations"] == 0 for r in reps)
    assert all(np.array_equal(r["pose"], r["T_ransac"]) for r in reps)


@pytest.mark.gpu
def test_gate_rejection_equals_chain(bshot, synth):
    """rotation 8 after rotation 2 is a 3 m jump: the gate rejects it (T_est = T_ref), the map is updated anyway"""
    p = bshot.odom_default_params(top_k=600)
    reps = run_pair(bshot, [synth.make_lasers("hdl32e", k) for k in (0, 1, 2, 8)], p, "lasers")
    assert reps[-1]["should_update_map"] == 0 and reps[-1]["t_diff_mm"] > 1200.0


@pytest.mark.gpu
def test_failed_step_leaves_state(bshot, synth):
    """a step whose target set overflows max_targets returns BSHOT_E_CAPACITY and changes neither pose, map nor reference
    frame: the next step gives exactly what it gives on a context that never failed"""
    small, large = 5000.0, 100000.0
    p_small = bshot.odom_default_params(top_k=600, map_range=small)
    p_large = bshot.odom_default_params(top_k=600, map_range=large)
    rot = [synth.make_lasers("hdl32e", k) for k in range(5)]

    def step(ctx, k, p):
        L = rot[k]
        return ctx.odometry_step(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p)

    # probe: how many map entries the two ranges gather before step 3
    with bshot.Context(0, 131072, 1024, 1 << 16) as c:
        c.gmap_create(1 << 16, 4096)
        for k in range(3):
            r = step(c, k, p_small)
        pos = r["pose"][:3, 3]
        n_small, n_large = len(c.gmap_get_keypoints(pos, small)[0]), len(c.gmap_get_keypoints(pos, large)[0])
    max_targets = max(n_small + 600, 1024)
    assert n_large + 600 > max_targets, (n_small, n_large)
    with bshot.Context(0, 131072, 1024, max_targets) as a, bshot.Context(0, 131072, 1024, max_targets) as b:
        for ctx in (a, b):
            ctx.gmap_create(1 << 16, 4096)
            for k in range(3):
                step(ctx, k, p_small)
        before = b.gmap_size()
        with pytest.raises(bshot.BshotError) as e:
            step(b, 3, p_large)
        assert e.value.code == bshot.E_CAPACITY
        assert b.gmap_size() == before
        for k in (3, 4):
            ra, rb = step(a, k, p_small), step(b, k, p_small)
            assert_same_report(rb, ra, k)
            assert a.gmap_size() == b.gmap_size()


@pytest.mark.gpu
def test_errors_and_reset(bshot, synth):
    L = synth.make_lasers("hdl32e", 0)
    p = bshot.odom_default_params(top_k=600)
    with bshot.Context(0, 131072, 1024, 1 << 16) as ctx:
        with pytest.raises(bshot.BshotError) as e:   # no map
            ctx.odometry_step(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p)
        assert e.value.code == bshot.E_STATE
        ctx.gmap_create(1 << 16, 4096)
        r = bshot.OdomReport()
        az = np.ascontiguousarray(L["azimuth"], np.float64)
        assert bshot.lib().bshot_odometry_step(ctx.h, C.byref(p), None, None, None, az.size, None, 0, C.byref(r)) == bshot.E_INVALID
        assert bshot.lib().bshot_odometry_step_cloud(ctx.h, C.byref(p), None, 100, 12, C.byref(r)) == bshot.E_INVALID
        for bad in (dict(ransac_iterations=0), dict(map_range=float("nan")), dict(inlier_threshold=-1.0)):
            with pytest.raises(bshot.BshotError) as e:
                ctx.odometry_step(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], bshot.odom_default_params(top_k=600, **bad))
            assert e.value.code == bshot.E_INVALID, bad
        rot = [synth.make_lasers("hdl32e", k) for k in range(4)]
        runs = []
        for _ in range(2):
            runs.append([ctx.odometry_step(x["azimuth"], x["vertical"], x["distance"], x["ring_deg"], p) for x in rot])
            runs[-1].append(ctx.gmap_size())
            ctx.odometry_reset()
            assert ctx.gmap_size() == (0, 0)
        for ra, rb in zip(runs[0][:-1], runs[1][:-1]):
            assert_same_report(rb, ra)
            assert np.float32(ra["h_diff_rad"]).view(np.uint32) == np.float32(rb["h_diff_rad"]).view(np.uint32)
        assert runs[0][-1] == runs[1][-1]


@pytest.mark.gpu
def test_device_odometry_shim_equals_python(bshot, synth, odometry_shim_binary, tmp_path):
    ring, paths, lasers = _write_rotations(tmp_path, synth, [0, 1, 2])
    out = str(tmp_path / "out.bin")
    r = subprocess.run([odometry_shim_binary, ring, out] + paths, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = np.fromfile(out, np.uint8).reshape(3, 80)
    p = bshot.odom_default_params()
    with bshot.Context(0, 131072, 1024, 1 << 16) as ctx:
        ctx.gmap_create(1 << 16, 4096)
        for k, L in enumerate(lasers):
            s = ctx.odometry_step(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p)
            pose = raw[k, :64].view(np.float32).reshape(4, 4)
            fields = raw[k, 64:].view(np.int32)
            assert np.array_equal(pose.view(np.uint32), s["pose"].view(np.uint32)), k
            assert list(fields) == [s["n_keypoints"], s["n_pairs"], s["n_inliers"], s["was_initial"]], k


# ---- GPU: bshot_ransac_dev against bshot_ransac ------------------------------------------------------------------------------
def _mt19937(seed):
    s = [0] * 624
    s[0] = seed
    for i in range(1, 624):
        s[i] = (1812433253 * (s[i - 1] ^ (s[i - 1] >> 30)) + i) & 0xFFFFFFFF
    idx = 624
    while True:
        if idx >= 624:
            for i in range(624):
                y = (s[i] & 0x80000000) | (s[(i + 1) % 624] & 0x7FFFFFFF)
                s[i] = s[(i + 397) % 624] ^ (y >> 1) ^ (0x9908B0DF if y & 1 else 0)
            idx = 0
        y = s[idx]
        idx += 1
        y ^= y >> 11
        y ^= (y << 7) & 0x9D2C5680
        y ^= (y << 15) & 0xEFC60000
        y ^= y >> 18
        yield y


def _hypotheses_before_giveup(labels, n_hyp):
    """PCL's sampler where a triple is good iff its three sources carry distinct labels (true for well separated groups):
    the number of hypotheses drawn before the 1000-try give-up (n_hyp = never gave up)"""
    n = len(labels)
    sh = list(range(n))
    rng = _mt19937(12345)
    for h in range(n_hyp):
        for _ in range(1000):
            for i in range(3):
                j = i + (next(rng) >> 1) % (n - i)
                sh[i], sh[j] = sh[j], sh[i]
            if len({labels[sh[0]], labels[sh[1]], labels[sh[2]]}) == 3:
                break
        else:
            return h
    return n_hyp


def _ransac_case(n, outliers, seed):
    rng = np.random.default_rng(seed)
    src = rng.uniform(-40000, 40000, (n, 3)).astype(np.float32)
    a = rng.uniform(-0.2, 0.2)
    R = np.array([[math.cos(a), -math.sin(a), 0], [math.sin(a), math.cos(a), 0], [0, 0, 1]])
    tgt = (src @ R.T + rng.uniform(-2000, 2000, 3) + rng.normal(0, 200, (n, 3))).astype(np.float32)
    bad = rng.random(n) < outliers
    tgt[bad] = rng.uniform(-40000, 40000, (int(bad.sum()), 3)).astype(np.float32)
    perm = rng.permutation(n).astype(np.int32)
    pairs = np.stack([np.arange(n, dtype=np.int32), perm], 1)
    tgt_p = np.empty_like(tgt)
    tgt_p[perm] = tgt
    return src, tgt_p, pairs


def _compare_ransac(ctx, src, tgt, pairs, max_iterations=2000, threshold=1500.0, cap=None):
    import torch
    host = ctx.ransac(src, tgt, pairs, max_iterations, threshold)
    s4 = torch.from_numpy(np.concatenate([src, np.ones((len(src), 1), np.float32)], 1)).cuda()
    t4 = torch.from_numpy(np.concatenate([tgt, np.ones((len(tgt), 1), np.float32)], 1)).cuda()
    cap = len(pairs) if cap is None else cap
    pp = np.zeros((max(cap, 1), 2), np.int32)
    pp[:len(pairs)] = pairs
    dev = ctx.ransac_dev(s4, t4, torch.from_numpy(pp).cuda(), torch.tensor([len(pairs)], dtype=torch.int32).cuda(), max_iterations, threshold)
    m = int(dev["n_inliers"].item())
    assert m == len(host["pairs"])
    assert np.array_equal(dev["pairs"].cpu().numpy()[:m], host["pairs"])
    assert np.array_equal(dev["transform"].cpu().numpy().view(np.uint32), host["transform"].view(np.uint32))
    assert int(dev["iterations"].item()) == host["iterations"]
    return host


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 4, 600, 5000])
@pytest.mark.parametrize("outliers", [0.0, 0.3, 0.6, 0.9])
def test_ransac_dev_equals_host(bshot, n, outliers):
    with bshot.Context(0, 1024, 8192, 8192) as ctx:
        src, tgt, pairs = _ransac_case(n, outliers, 17 + n)
        _compare_ransac(ctx, src, tgt, pairs)
        _compare_ransac(ctx, src, tgt, pairs, cap=n + 37)   # a capacity past the device-side count


@pytest.mark.gpu
def test_ransac_dev_sampler_cases(bshot):
    rng = np.random.default_rng(5)
    with bshot.Context(0, 1024, 8192, 8192) as ctx:
        # clustered sources: most triples hold two points of the cluster and are retried
        src = np.concatenate([rng.normal(0, 1.0, (400, 3)), rng.uniform(-30000, 30000, (200, 3))]).astype(np.float32)
        tgt = (src + np.float32([700, -300, 50])).astype(np.float32)
        pairs = np.stack([np.arange(600), np.arange(600)], 1).astype(np.int32)
        r = _compare_ransac(ctx, src, tgt, pairs)
        assert r["iterations"] > 0
        # all sources identical: no sample can be drawn, everything is kept with the identity
        same = np.tile(np.float32([[1000, 2000, 3000]]), (300, 1))
        pairs = np.stack([np.arange(300), np.arange(300)], 1).astype(np.int32)
        r = _compare_ransac(ctx, same, same + np.float32(5), pairs)
        assert r["iterations"] == 0 and len(r["pairs"]) == 300 and np.array_equal(r["transform"], np.eye(4, dtype=np.float32))
        # a few distinct points among a large cluster: the give-up fires after some hypotheses, before the last
        n_distinct, n = 20, 600
        labels = list(range(1, n_distinct + 1)) + [0] * (n - n_distinct)
        n_valid = _hypotheses_before_giveup(labels, 2001)
        assert 0 < n_valid < 2001, n_valid
        pts = np.zeros((n, 3), np.float32)   # the cluster at the origin, the distinct points on a 30 m lattice away from it
        i = np.arange(n_distinct)
        pts[:n_distinct] = 30000.0 * np.stack([1 + i % 3, 1 + (i // 3) % 3, 1 + i // 9], 1)
        tgt = pts + np.float32([300, 0, 0])
        tgt[n_distinct:] = rng.uniform(-50000, 50000, (n - n_distinct, 3)).astype(np.float32)   # the cluster's targets are outliers
        pairs = np.stack([np.arange(n), np.arange(n)], 1).astype(np.int32)
        _compare_ransac(ctx, pts, tgt, pairs)   # (every good triple holds an outlier pair here: PCL keeps everything)
        tgt[n_distinct:] = pts[n_distinct:] + np.float32([300, 0, 0])
        _compare_ransac(ctx, pts, tgt, pairs)   # the same sample sequence with consistent targets
