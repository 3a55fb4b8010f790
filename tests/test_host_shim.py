"""The reference-named host C++ layer (b-shot-slam_b200/host/*.h: bshot, bshot_descriptor, minVect,
Frame, Keypoint, Map, LidarOdometry stage methods) compiled with g++ against the C-ABI library.
CPU: it compiles/links and fails loudly without a GPU.  GPU: the reference's call order
(test/odometry_test.cpp:174-180) on two frames, checked against the oracle."""
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "b-shot-slam_b200")
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from snapshots import ExpectedPreprocessing, Snapshots  # noqa: E402


@pytest.fixture(scope="module")
def shim_binary(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("shim") / "host_shim_test")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror",
                           os.path.join(ROOT, "tests", "host_shim_test.cpp"), "-o", out, "-L", PKG, "-lbshot_b200",
                           f"-Wl,-rpath,{PKG}"])
    return out


def test_shims_compile_and_fail_loudly_without_gpu(shim_binary):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([shim_binary, "a", "b", "c"], capture_output=True, text=True)
    assert r.returncode == 1 and "no CPU fallback" in r.stdout


@pytest.mark.gpu
def test_reference_call_order_two_frames(shim_binary, tmp_path, oracle, synth, gpu_ctx):
    scans = [synth.make_scan("hdl32e", f)[::2].copy() for f in (0, 1)]
    paths = []
    for i, s in enumerate(scans):
        p = str(tmp_path / f"cloud{i}.bin")
        s.tofile(p)
        paths.append(p)
    outp = str(tmp_path / "out.bin")
    L = synth.make_lasers("hdl32e", 0, firings=500, start_deg=300.0)
    lasers, pre_out = str(tmp_path / "lasers.bin"), str(tmp_path / "pre.bin")
    with open(lasers, "wb") as fh:
        fh.write(L["azimuth"].tobytes() + L["vertical"].tobytes() + L["distance"].tobytes())
    r = subprocess.run([shim_binary, paths[0], paths[1], outp, lasers, pre_out], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    # myslam::Preprocessor shim == the reference's preprocess.cpp compiled unchanged where it is built, and everywhere
    # the regression snapshot of the device preprocessor (tests/golden/snapshots.py)
    got = np.fromfile(pre_out, np.float32).reshape(-1, 3)
    snapshots = Snapshots()
    want = ExpectedPreprocessing(snapshots, oracle, gpu_ctx).preprocess(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"])
    snapshots.save()
    want.check(got, "preprocessed points")
    raw = open(outp, "rb").read()
    off, frames, rest = 0, [], []
    for _ in range(2):
        k, nc = struct.unpack_from("ii", raw, off); off += 8
        kp = np.frombuffer(raw, np.float32, 3 * k, off).reshape(k, 3); off += 12 * k
        bits = np.frombuffer(raw, np.uint64, 6 * k, off).reshape(k, 6); off += 48 * k
        rf = np.frombuffer(raw, np.float32, 9 * k, off).reshape(k, 9); off += 36 * k
        corr = np.frombuffer(raw, np.int32, 2 * nc, off).reshape(nc, 2); off += 8 * nc
        nt, = struct.unpack_from("i", raw, off); off += 4
        tgt = np.frombuffer(raw, np.uint64, 6 * nt, off).reshape(nt, 6); off += 48 * nt
        tgt_xyz = np.frombuffer(raw, np.float32, 3 * nt, off).reshape(nt, 3); off += 12 * nt
        nr, = struct.unpack_from("i", raw, off); off += 4
        kept = np.frombuffer(raw, np.int32, 2 * nr, off).reshape(nr, 2); off += 8 * nr
        upd, = struct.unpack_from("i", raw, off); off += 4
        T_ransac = np.frombuffer(raw, np.float32, 16, off).reshape(4, 4); off += 64
        pose = np.frombuffer(raw, np.float32, 16, off).reshape(4, 4); off += 64
        frames.append((kp, bits, rf, corr, tgt))
        rest.append((tgt_xyz, kept, upd, T_ransac, pose))
    assert off == len(raw)
    assert "same-size reassignment ok" in r.stdout
    for (kp, bits, rf, corr, _), scan in zip(frames, scans):
        assert len(kp) == 600                                   # reference default K (src/lidar_odometry.cpp:138)
        oc = oracle.Cloud(scan)
        od = oc.compute_descriptors(kp, 3000.0, 300, oracle.MODE_REFERENCE)
        ok = ~np.isnan(od["rf"]).any(1)
        assert np.abs(rf[ok] - od["rf"][ok]).max() <= 1e-4
        assert (synth.unpack_bits(bits) == synth.unpack_bits(od["bits"])).mean() >= 0.999
    # frame 0 matched against itself (:187-194); frame 1 against (map keypoints within 100 m) + the reference frame's
    # descriptors (:197-206): the shim dumps the target set it assembled, the correspondences must be exactly the
    # oracle's mutual nearest neighbours on it
    (_, b0, _, c0, t0), (_, b1, _, c1, t1) = frames
    assert np.array_equal(t0, b0)
    m = oracle.match(b0, t0)
    assert np.array_equal(c0, oracle.mutual(m["left_idx"], m["right_idx"]))
    assert len(t1) > 600 and np.array_equal(t1[-600:], b0)      # map subset first, then the 600 reference-frame records
    m1 = oracle.match(b1, t1)
    assert len(c1) > 0 and np.array_equal(c1, oracle.mutual(m1["left_idx"], m1["right_idx"]))
    # RANSAC rejection, the gate + ICP and the pose (featureMatching :251-261, evaluateEstimation, poseEstimation):
    # the oracle on the same keypoints / correspondences gives the same bits
    pose_ref = np.eye(4, dtype=np.float32)
    for (kp, _, _, c, _), (tgt_xyz, kept, upd, T_ransac, pose) in zip(frames, rest):
        rs = oracle.ransac(kp, tgt_xyz, c)
        assert np.array_equal(kept, rs["pairs"]) and np.array_equal(T_ransac, rs["transform"])
        ev = oracle.evaluate_estimation(rs["transform"], pose_ref, len(rs["pairs"]), kp, tgt_xyz, run_icp=True)
        assert bool(upd) == ev["should_update_map"]
        assert np.array_equal(pose.view(np.uint32), ev["T_best"].view(np.uint32))
        pose_ref = pose
