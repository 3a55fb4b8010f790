"""ctypes binding of tests/iss_oracle.cpp: the CPU restatement of the ISS detector and of the keypoint repeatability
measure (test infrastructure; the parity pin is described at the top of iss_oracle.cpp).  The source is compiled once
per process into a temporary directory, against the CPU oracle's library (oracle/libbshot_oracle.so), so the tree is
never written to."""
import ctypes as C
import os
import subprocess
import sys
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_LIB = None


def _oracle():
    sys.path.insert(0, _HERE)
    from conftest import load_oracle
    return load_oracle()


def lib():
    global _LIB
    if _LIB is None:
        oracle_so = _oracle().build()            # oracle/libbshot_oracle.so, built by build() / make -C oracle
        odir = os.path.dirname(oracle_so)
        out = os.path.join(tempfile.mkdtemp(prefix="iss_oracle_"), "libiss_oracle.so")
        subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O3", "-march=x86-64-v3", "-ffp-contract=off", "-fopenmp", "-fPIC",
                               "-Wall", "-Wextra", "-shared", "-I", os.path.join(_ROOT, "oracle"), os.path.join(_HERE, "iss_oracle.cpp"),
                               "-L", odir, "-lbshot_oracle", f"-Wl,-rpath,{odir}", "-o", out])
        L = C.CDLL(out)
        fp, ip, dp = C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_double)
        L.iss_ref_detect.restype = C.c_int
        L.iss_ref_detect.argtypes = [C.c_void_p, fp, C.c_size_t, C.c_float, C.c_float, C.c_double, C.c_double, C.c_int, C.c_int, ip,
                                     C.c_size_t, dp]
        L.iss_ref_repeatability.restype = C.c_size_t
        L.iss_ref_repeatability.argtypes = [fp, C.c_size_t, fp, fp, C.c_size_t, fp, C.c_float, ip, fp]
        _LIB = L
    return _LIB


def _f(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_float))


def iss(cloud, salient_radius=60.0, non_max_radius=40.0, gamma_21=0.975, gamma_32=0.975, min_neighbors=5, threads=0,
        want_eigs=False):
    """pcl::ISSKeypoint3D as issKpDetection calls it (src/lidar_odometry.cpp:447-461) on a pyoracle.Cloud: keypoint
    indices ascending (and the N x 3 eigenvalues l1..l3 when want_eigs)"""
    n = len(cloud)
    idx = np.empty(max(n, 1), np.int32)
    eigs = np.empty((n, 3), np.float64) if want_eigs else None
    k = lib().iss_ref_detect(cloud.h, _f(cloud.xyz), n, salient_radius, non_max_radius, gamma_21, gamma_32, min_neighbors, threads,
                             idx.ctypes.data_as(C.POINTER(C.c_int)), n,
                             None if eigs is None else eigs.ctypes.data_as(C.POINTER(C.c_double)))
    return (idx[:k].copy(), eigs) if want_eigs else idx[:k].copy()


def _pose12(pose):
    if pose is None:
        return None
    m = np.asarray(pose, dtype=np.float32)
    if m.size == 16:
        m = m.reshape(4, 4)[:3]
    return np.ascontiguousarray(m.reshape(12))


def kp_repeatability(a, b, pose_a=None, pose_b=None, radius=30.0):
    """kpEvaluation (src/lidar_odometry.cpp:392-445), the port's definition: nearest point of B (moved by pose_b) for every
    point of A (moved by pose_a) -> dict(nn_idx, nn_dist, hits, rate)"""
    a = np.ascontiguousarray(a, dtype=np.float32).reshape(-1, 3)
    b = np.ascontiguousarray(b, dtype=np.float32).reshape(-1, 3)
    pa, pb = _pose12(pose_a), _pose12(pose_b)
    na = a.shape[0]
    idx = np.empty(max(na, 1), np.int32)
    dist = np.empty(max(na, 1), np.float32)
    hits = lib().iss_ref_repeatability(_f(a), na, _f(pa), _f(b), b.shape[0], _f(pb), radius, idx.ctypes.data_as(C.POINTER(C.c_int)),
                                       _f(dist))
    return dict(nn_idx=idx[:na].copy(), nn_dist=dist[:na].copy(), hits=int(hits), rate=hits / na if na else 0.0)
