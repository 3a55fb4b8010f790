"""Voxel-grid downsampling (pcl::VoxelGrid<PointXYZ> as the reference's bshot::calculate_voxel_grid_keypoints calls it).
CPU: known answers of the reference (tests/voxel_grid_oracle.cpp), an independent numpy restatement, and PCL's unstable
within-voxel order against the port's ascending point index.  GPU: bshot_voxel_grid against the reference bit for bit,
errors, no side effects on the frame path, voxel centroids through B-SHOT, and the host shim."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

import voxel_grid_oracle as vgo  # CPU restatement of pcl::VoxelGrid (tests/voxel_grid_oracle.cpp)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "b-shot-slam_b200")
LEAVES = [100.0, 500.0, 1000.0, 3000.0, (200.0, 200.0, 50.0)]
# voxels of the seeded frame-0 scans at leaves 100, 500, 1000, 3000 mm
EXPECTED_COUNTS = {"hdl64e": [95598, 33124, 16150, 2511], "hdl32e": [48479, 20141, 9684, 1789]}
NAN = np.float32(np.nan)


def _bits_equal(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _lattice():
    """two points in each of 3 x 2 x 2 voxels of a 100 mm grid, input in a scrambled order; centroids are exact"""
    pts, want = [], []
    for k in range(2):
        for j in range(2):
            for i in range(3):
                b = np.float32([100 * i, 100 * j, 100 * k])
                pts += [b + [10, 20, 30], b + [30, 40, 50]]
                want.append(b + [20, 30, 40])
    pts = np.array(pts, np.float32)
    perm = np.random.default_rng(3).permutation(len(pts))
    return pts[perm], np.array(want, np.float32)


def known_answers():
    """(name, cloud, leaf, expected output)"""
    lat, lat_want = _lattice()
    cases = [("lattice, x fastest", lat, 100.0, lat_want)]
    # floor, not truncation: -50 and -10 share bin -1, 10 is in bin 0
    cases.append(("negative coordinates", np.float32([[10, 10, 10], [-50, 10, 10], [-10, 10, 10]]), 100.0,
                  np.float32([[-30, 10, 10], [10, 10, 10]])))
    # 0.001f is slightly above 1/1000: -3000 * 0.001f = -3.0000001 -> bin -4, the same bin as -3500
    cases.append(("leaf 1000 fp32 product", np.float32([[-3000, 0, 0], [-3500, 0, 0]]), 1000.0, np.float32([[-3250, 0, 0]])))
    # anisotropic: 200 mm in x / y, 50 mm in z
    cases.append(("anisotropic leaf", np.float32([[10, 10, 60], [10, 10, 10], [150, 150, 40], [250, 10, 10]]), (200.0, 200.0, 50.0),
                  np.float32([[80, 80, 25], [250, 10, 10], [10, 10, 60]])))
    # -0.0 is the largest x here and lies in bin 0; -50 and -60 share bin -1
    cases.append(("negative zero", np.float32([[-0.0, 0, 0], [-50, 0, 0], [-60, 0, 0]]), 100.0,
                  np.float32([[-55, 0, 0], [0, 0, 0]])))
    cases.append(("one point", np.float32([[123.5, -7.25, 3.0]]), 100.0, np.float32([[123.5, -7.25, 3.0]])))
    bad = np.float32([[NAN, 0, 0], [0, np.inf, 0], [1, 2, -np.inf]])
    cases.append(("non-finite points skipped", np.insert(lat, [0, 5, 24], bad, axis=0), 100.0, lat_want))
    cases.append(("all non-finite", bad, 100.0, np.zeros((0, 3), np.float32)))
    cases.append(("empty", np.zeros((0, 3), np.float32), 100.0, np.zeros((0, 3), np.float32)))
    return cases


def negative_zero_tiles():
    """3072 points in three tiles of 1024 (the device's bbox tiles): x is -0.0 in tile 0 and negative elsewhere, z is
    -0.0 in tile 1 and negative elsewhere, so one tile's min and the cloud's max of those axes are -0.0"""
    rng = np.random.default_rng(11)
    P = np.empty((3072, 3), np.float32)
    P[:, 0] = rng.uniform(-5000.0, -10.0, 3072)
    P[:, 1] = rng.uniform(-3000.0, 3000.0, 3072)
    P[:, 2] = rng.uniform(-800.0, -5.0, 3072)
    P[:1024, 0] = -0.0
    P[1024:2048, 2] = -0.0
    return P


def overflow_cloud(synth):
    """an HDL-32E scan with a NaN point: at leaf 1 mm the grid has more than INT32_MAX cells"""
    return np.insert(synth.make_scan("hdl32e", 0), 17, [NAN, 1.0, 2.0], axis=0)


def numpy_voxel_grid(xyz, leaf):
    """independent restatement: fp32 products, np.floor, lexsort on (voxel index, point index), per-voxel
    np.add.accumulate in float32.  Returns (centroids, voxel of every sorted point, sorted points) or the input on
    overflow"""
    xyz = np.asarray(xyz, np.float32)[:, :3]
    inv = np.float32(1.0) / np.float32(vgo.leaf3(leaf))
    fin = np.isfinite(xyz).all(1)
    P = xyz[fin]
    if len(P) == 0:
        return np.zeros((0, 3), np.float32), None, None
    mn, mx = P.min(0), P.max(0)
    d = ((mx - mn) * inv).astype(np.int64) + 1
    if int(d[0]) * int(d[1]) * int(d[2]) > 2**31 - 1:
        return xyz.copy(), None, None
    min_b = np.floor(mn * inv).astype(np.int64)
    div = np.floor(mx * inv).astype(np.int64) - min_b + 1
    mul = np.array([1, div[0], div[0] * div[1]], np.int64)
    ijk = (np.floor(P * inv) - min_b.astype(np.float32)).astype(np.int64)
    idx = (ijk @ mul) % (1 << 32)
    order = np.lexsort((np.nonzero(fin)[0], idx))
    sidx, sp = idx[order], P[order]
    starts = np.flatnonzero(np.r_[True, sidx[1:] != sidx[:-1]])
    ends = np.r_[starts[1:], len(sidx)]
    out = np.empty((len(starts), 3), np.float32)
    for v, (s, e) in enumerate(zip(starts, ends)):
        # the sum starts from +0 as PCL's centroid.setZero() (a voxel of -0.0 coordinates sums to +0)
        acc = np.add.accumulate(np.vstack([np.zeros((1, 3), np.float32), sp[s:e]]), axis=0, dtype=np.float32)
        out[v] = acc[-1] / np.float32(e - s)
    seg = np.repeat(np.arange(len(starts)), ends - starts)
    return out, seg, sp


def pcl_order_bound(ref, seg, sp):
    """per component bound of |pcl - index|: 2 (m - 1) 2^-24 sum|x_i| / m + 2 ulp"""
    m = np.bincount(seg).astype(np.float64)[:, None]
    sabs = np.zeros((len(m), 3))
    np.add.at(sabs, seg, np.abs(sp.astype(np.float64)))
    return 2.0 * (m - 1) * 2.0**-24 * sabs / m + 2.0 * np.spacing(np.abs(ref)).astype(np.float64)


def check_pcl_order(xyz, leaf, got, what):
    """the "pcl" order (std::sort) gives the same voxels in the same order as `got`, centroids within the bound"""
    ref, seg, sp = numpy_voxel_grid(xyz, leaf)
    pcl = vgo.voxel_grid(xyz, leaf, "pcl")
    assert pcl.shape == got.shape, what
    diff = np.abs(pcl.astype(np.float64) - got.astype(np.float64))
    assert (diff <= pcl_order_bound(ref, seg, sp)).all(), what
    n_diff = int((diff > 0).any(1).sum())
    print(f"{what}: {len(got)} voxels, {n_diff} differ between the pcl and index orders")
    return n_diff


# ---- CPU: the restatement (tests/voxel_grid_oracle.cpp) ----------------------------------------------------------------
@pytest.mark.parametrize("case", known_answers(), ids=lambda c: c[0])
def test_cpu_voxel_grid_known_answers(case):
    _, xyz, leaf, want = case
    assert _bits_equal(vgo.voxel_grid(xyz, leaf), want)
    assert _bits_equal(vgo.voxel_grid(xyz, leaf, "pcl"), want)


def test_cpu_voxel_grid_fp32_binning():
    # the case above needs the fp32 product: a division (or double arithmetic) puts -3000 in bin -3, apart from -3500
    assert np.floor(np.float32(-3000) * (np.float32(1) / np.float32(1000))) == -4.0
    assert np.floor(-3000 / 1000.0) == -3.0


def test_cpu_voxel_grid_overflow_copies_the_input(synth):
    xyz = overflow_cloud(synth)
    out = vgo.voxel_grid(xyz, 1.0)
    assert _bits_equal(out, xyz) and np.isnan(out[17, 0])
    assert len(vgo.voxel_grid(xyz, 100.0)) < len(xyz)     # the same scan does not overflow at 100 mm


def test_cpu_voxel_grid_negative_zero_tiles():
    xyz = negative_zero_tiles()
    got = vgo.voxel_grid(xyz, 100.0)
    want, _, _ = numpy_voxel_grid(xyz, 100.0)
    assert len(got) > 1000 and _bits_equal(got, want)
    assert np.signbit(xyz[:1024, 0]).all() and got[:, 0].max() == 0.0


def test_cpu_voxel_grid_stride16():
    xyz, want = _lattice()
    xyz4 = np.hstack([xyz, np.full((len(xyz), 1), 7.0, np.float32)])
    assert _bits_equal(vgo.voxel_grid(xyz4, 100.0), want)


@pytest.mark.parametrize("sensor", ["hdl32e", "hdl64e"])
def test_cpu_voxel_grid_matches_numpy_restatement(synth, sensor):
    xyz = synth.make_scan(sensor, 0)
    for k, leaf in enumerate(LEAVES):
        got = vgo.voxel_grid(xyz, leaf)
        want, _, _ = numpy_voxel_grid(xyz, leaf)
        assert _bits_equal(got, want), (sensor, leaf)
        if k < 4:
            assert len(got) == EXPECTED_COUNTS[sensor][k], (sensor, leaf, len(got))


@pytest.mark.parametrize("sensor", ["hdl32e", "hdl64e"])
def test_cpu_voxel_grid_pcl_order_within_bound(synth, sensor):
    xyz = synth.make_scan(sensor, 0)
    for leaf in LEAVES:
        check_pcl_order(xyz, leaf, vgo.voxel_grid(xyz, leaf), f"{sensor} leaf {leaf}")


# ---- GPU: bshot_voxel_grid ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("sensor", ["hdl32e", "hdl64e"])
@pytest.mark.parametrize("leaf", LEAVES, ids=str)
def test_voxel_grid_parity(synth, gpu_ctx, sensor, leaf):
    xyz = synth.make_scan(sensor, 0)
    got = gpu_ctx.voxel_grid(xyz, leaf)
    assert _bits_equal(got, vgo.voxel_grid(xyz, leaf)), (sensor, leaf)
    check_pcl_order(xyz, leaf, got, f"device {sensor} leaf {leaf}")


@pytest.mark.gpu
def test_voxel_grid_known_answers(synth, gpu_ctx):
    for name, xyz, leaf, want in known_answers():
        assert _bits_equal(gpu_ctx.voxel_grid(xyz, leaf), want), name
    xyz, want = _lattice()
    assert _bits_equal(gpu_ctx.voxel_grid(np.hstack([xyz, np.ones((len(xyz), 1), np.float32)]), 100.0), want)  # stride 16
    xyz = overflow_cloud(synth)
    assert _bits_equal(gpu_ctx.voxel_grid(xyz, 1.0), xyz)


@pytest.mark.gpu
@pytest.mark.parametrize("leaf", [100.0, 1000.0], ids=str)
def test_voxel_grid_negative_zero_tiles(gpu_ctx, leaf):
    xyz = negative_zero_tiles()
    for _ in range(3):                                                    # tiles may reach the bbox in any order
        assert _bits_equal(gpu_ctx.voxel_grid(xyz, leaf), vgo.voxel_grid(xyz, leaf))


@pytest.mark.gpu
def test_grid_build_with_negative_zero_extremes(gpu_ctx, oracle):
    """the frame path's voxel table uses the same float atomics for its bounding box: a cloud whose x max and one
    tile's x min are -0.0 gives the seg-ratios of the CPU oracle"""
    xyz = negative_zero_tiles()
    xyz[:, 0] *= 1.2
    gpu_ctx.set_cloud(xyz)
    rg = gpu_ctx.seg_ratio(1500.0, 50, 0)
    ro = oracle.Cloud(xyz).seg_ratio(1500.0, 50, oracle.SR_CV)
    assert np.array_equal(np.isnan(rg), np.isnan(ro))
    ok = ~np.isnan(ro)
    assert ok.sum() > 3000 and np.array_equal(rg[ok], ro[ok])


@pytest.mark.gpu
def test_voxel_grid_one_voxel_holds_the_whole_cloud(synth, gpu_ctx):
    xyz = synth.make_scan("hdl64e", 0)
    xyz = (xyz - xyz.min(0) + np.float32(1000.0)).astype(np.float32)   # every coordinate in [1000, 202000] mm
    got = gpu_ctx.voxel_grid(xyz, 1.0e6)
    assert got.shape == (1, 3) and _bits_equal(got, vgo.voxel_grid(xyz, 1.0e6))
    check_pcl_order(xyz, 1.0e6, got, "one voxel")


@pytest.mark.gpu
def test_voxel_grid_repeatable(synth, gpu_ctx):
    xyz = synth.make_scan("hdl64e", 1)
    a = gpu_ctx.voxel_grid(xyz, 500.0)
    b = gpu_ctx.voxel_grid(xyz, 500.0)
    assert _bits_equal(a, b)


@pytest.mark.gpu
def test_voxel_grid_capacity_and_arguments(bshot, synth):
    L = bshot.lib()
    cnt = C.c_size_t()
    with bshot.Context(0, 65536, 1024, 1024) as ctx:
        xyz = synth.make_scan("hdl32e", 0)[:60000].copy()
        for bad in ((0.0, 1.0, 1.0), (1.0, -1.0, 1.0), (1.0, 1.0, float("nan")), (float("inf"), 1.0, 1.0), (1e-40, 1.0, 1.0)):
            assert L.bshot_voxel_grid(ctx.h, bshot._p(xyz), len(xyz), 12, *bad, None, 0, C.byref(cnt)) == -1, bad
        assert L.bshot_voxel_grid(ctx.h, None, 10, 12, 100.0, 100.0, 100.0, None, 0, C.byref(cnt)) == -1
        assert L.bshot_voxel_grid(ctx.h, bshot._p(xyz), len(xyz), 8, 100.0, 100.0, 100.0, None, 0, C.byref(cnt)) == -1
        big = synth.make_scan("hdl64e", 0)                                  # 120 000 > max_points
        assert L.bshot_voxel_grid(ctx.h, bshot._p(big), len(big), 12, 100.0, 100.0, 100.0, None, 0, C.byref(cnt)) == bshot.E_CAPACITY
        full = ctx.voxel_grid(xyz, 500.0)
        k = len(full)
        assert k == len(vgo.voxel_grid(xyz, 500.0)) and k > 1000
        cap = k // 3
        out = np.full((k, 3), -7.0, np.float32)
        rc = L.bshot_voxel_grid(ctx.h, bshot._p(xyz), len(xyz), 12, 500.0, 500.0, 500.0, bshot._p(out), cap, C.byref(cnt))
        assert rc == bshot.E_CAPACITY and cnt.value == k
        assert _bits_equal(out[:cap], full[:cap]) and (out[cap:] == -7.0).all()
        assert L.bshot_voxel_grid(ctx.h, None, 0, 12, 100.0, 100.0, 100.0, None, 0, C.byref(cnt)) == 0 and cnt.value == 0


def _frame_loop(bshot, synth, with_vg, process_frame=False):
    """four frames through the frame-to-map flow (or bshot_process_frame), optionally with voxel-grid calls on another
    scan after the extraction; returns everything the loop produced"""
    p = bshot.default_params(top_k=600)
    other = synth.make_scan("hdl64e", 2)
    out = []
    with bshot.Context(0, 131072, 1024, 1 << 15) as ctx:
        if process_frame:
            for k in range(4):
                f = ctx.process_frame(synth.make_scan("hdl32e", k), p)
                if with_vg:
                    ctx.voxel_grid(other, 300.0)
                out += [f["kp_idx"], f["bits"], f["pairs"]]
            return out
        ctx.gmap_create(1 << 15, 4096)
        pose = np.eye(4, dtype=np.float32)[:3].copy()
        for k in range(4):
            f = ctx.extract_frame(synth.make_scan("hdl32e", k), p)
            if with_vg:
                ctx.voxel_grid(other, 300.0)
                ctx.voxel_grid(other, 1.0)                                # the overflow copy too
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
def test_voxel_grid_has_no_side_effects(bshot, synth, process_frame):
    a = _frame_loop(bshot, synth, False, process_frame)
    b = _frame_loop(bshot, synth, True, process_frame)
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8))


@pytest.mark.gpu
def test_voxel_keypoints_through_bshot(bshot, oracle, synth, gpu_ctx):
    xyz = synth.make_scan("hdl64e", 0)
    kp = gpu_ctx.voxel_grid(xyz, 3000.0)
    assert len(kp) == EXPECTED_COUNTS["hdl64e"][3]
    gpu_ctx.set_cloud(xyz)
    gpu_ctx.set_keypoints(kp)
    bits = gpu_ctx.compute_descriptors(bshot.default_params())
    od = oracle.Cloud(xyz).compute_descriptors(kp, 3000.0, 300, oracle.MODE_REFERENCE)
    same = (synth.unpack_bits(bits) == synth.unpack_bits(od["bits"])).mean()
    print(f"voxel keypoints through B-SHOT: {len(kp)} keypoints, {same:.6f} of the bits identical")
    assert same >= 0.999, same


@pytest.fixture(scope="module")
def voxel_shim_binary(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("voxel_shim") / "host_shim_voxel_test")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror",
                           os.path.join(ROOT, "tests", "host_shim_voxel_test.cpp"), "-o", out, "-L", PKG, "-lbshot_b200",
                           f"-Wl,-rpath,{PKG}"])
    return out


def test_voxel_shim_compiles(voxel_shim_binary):
    assert os.path.exists(voxel_shim_binary)


@pytest.mark.gpu
def test_voxel_shim_keypoints_and_descriptors(voxel_shim_binary, bshot, synth, tmp_path):
    """cb.calculate_voxel_grid_keypoints(leaf) on two clouds, then calculate_normals -> calculate_SHOT -> compute_bshot:
    the keypoints equal Context.voxel_grid of each cloud and the bits equal the Python chain's"""
    clouds = [synth.make_scan("hdl32e", 0), synth.make_scan("hdl64e", 1)]
    paths = []
    for i, c in enumerate(clouds):
        paths.append(str(tmp_path / f"cloud{i}.bin"))
        c.tofile(paths[-1])
    outp = str(tmp_path / "out.bin")
    leaf = 1500.0
    r = subprocess.run([voxel_shim_binary, paths[0], paths[1], str(leaf), outp], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = open(outp, "rb").read()
    off, kps = 0, []
    for _ in range(2):
        n, width, height, dense = struct.unpack_from("4i", raw, off); off += 16
        kps.append(np.frombuffer(raw, np.float32, 3 * n, off).reshape(n, 3)); off += 12 * n
        assert (width, height, dense) == (n, 1, 1)
    (nb,) = struct.unpack_from("i", raw, off); off += 4
    bits = np.frombuffer(raw, np.uint64, 6 * nb, off).reshape(nb, 6); off += 48 * nb
    assert off == len(raw)
    with bshot.Context(0, 1 << 18, 1 << 14, 1 << 10) as ctx:
        for k in range(2):
            assert _bits_equal(kps[k], ctx.voxel_grid(clouds[k], leaf))
        ctx.set_cloud(clouds[0])
        ctx.set_keypoints(kps[0])
        ctx.compute_normals(bshot.NORMALS_REFERENCE, 3000.0, 300)
        want = ctx.compute_shot(3000.0)["bits"]
    assert nb == len(kps[0]) > 0 and np.array_equal(bits, want)


@pytest.mark.gpu
def test_voxel_shim_overflow_copy_keeps_the_input_layout(voxel_shim_binary, synth, tmp_path):
    """PCL returns the input cloud itself when the grid would overflow, organized layout included; a result where every
    point sits alone in its voxel, in input order, is binned output all the same (height 1, dense)"""
    scan = synth.make_scan("hdl32e", 0)[:20000].copy()
    scan[5] = NAN
    alone = np.stack([1000.0 * np.arange(100) + 10.0, np.full(100, 10.0), np.full(100, 10.0)], 1).astype(np.float32)
    paths = [str(tmp_path / "scan.bin"), str(tmp_path / "alone.bin")]
    scan.tofile(paths[0])
    alone.tofile(paths[1])
    outp = str(tmp_path / "out.bin")
    r = subprocess.run([voxel_shim_binary, paths[0], paths[1], "1", outp, "organize"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = open(outp, "rb").read()
    off, got = 0, []
    for _ in range(2):
        n, width, height, dense = struct.unpack_from("4i", raw, off); off += 16
        got.append(((width, height, dense), np.frombuffer(raw, np.float32, 3 * n, off).reshape(n, 3))); off += 12 * n
    assert off == len(raw)
    assert got[0][0] == (len(scan) // 2, 2, 0) and _bits_equal(got[0][1], scan)        # the overflow copy
    assert got[1][0] == (len(alone), 1, 1) and _bits_equal(got[1][1], alone)           # binned, every point alone
