"""ctypes binding of tests/voxel_grid_oracle.cpp: the CPU restatement of pcl::VoxelGrid (test infrastructure; the
parity pin is described at the top of voxel_grid_oracle.cpp).  The source is compiled once per process into a temporary
directory, so the tree is never written to; it needs no other library."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
ORDERS = {"index": 0, "pcl": 1}


def lib():
    global _LIB
    if _LIB is None:
        out = os.path.join(tempfile.mkdtemp(prefix="voxel_grid_oracle_"), "libvoxel_grid_oracle.so")
        subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O3", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra", "-shared",
                               os.path.join(_HERE, "voxel_grid_oracle.cpp"), "-o", out])
        L = C.CDLL(out)
        L.vg_ref_filter.restype = C.c_size_t
        L.vg_ref_filter.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_float, C.c_float, C.c_float, C.c_int, C.c_void_p]
        _LIB = L
    return _LIB


def leaf3(leaf):
    """a scalar or a 3-sequence -> three float leaf sizes"""
    l3 = np.broadcast_to(np.asarray(leaf, dtype=np.float32), (3,))
    return tuple(float(v) for v in l3)


def voxel_grid(xyz, leaf, order="index"):
    """pcl::VoxelGrid<PointXYZ> (setLeafSize(leaf), filter) on an (N, 3) or (N, 4) float32 cloud -> (M, 3) float32"""
    xyz = np.ascontiguousarray(xyz, dtype=np.float32)
    assert xyz.ndim == 2 and xyz.shape[1] in (3, 4)
    n = xyz.shape[0]
    out = np.empty((max(n, 1), 3), np.float32)
    m = lib().vg_ref_filter(xyz.ctypes.data if n else None, n, xyz.shape[1], *leaf3(leaf), ORDERS[order], out.ctypes.data)
    return out[:m].copy()
