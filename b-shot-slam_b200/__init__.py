"""bshot_b200 -- Python (ctypes) binding of the B200-native B-SHOT front end.

The product is the C-ABI shared library `libbshot_b200.so` (include/bshot_b200.h) built from the
sm_100a CUDA sources in csrc/.  This module only marshals numpy / torch buffers to that ABI for the
tests and bench.py.  There is NO CPU fallback: if the library is missing or no B200 is present the
calls raise.  Reference-named host C++ shims live in host/ (see INTEGRATION.md).

The directory name `b-shot-slam_b200` is not an importable identifier; load this package with
`importlib` under the name `bshot_b200` (tests/conftest.py, bench.py and __graft_entry__.py do so).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BSHOT_LIB") or os.path.join(_HERE, "libbshot_b200.so")  # BSHOT_LIB: tuning builds (tools/build_variant.sh)
_LIB = None

SR_CV, SR_CVS, SR_CVSN = 0, 1, 2
NORMALS_REFERENCE, NORMALS_FULL = 0, 1

EXPORTS = [
    "bshot_params_default", "bshot_version", "bshot_last_error", "bshot_ctx_create",
    "bshot_ctx_destroy", "bshot_ctx_stream", "bshot_ctx_sync", "bshot_ctx_reset", "bshot_set_cloud",
    "bshot_detect_keypoints", "bshot_seg_ratio", "bshot_set_keypoints", "bshot_compute_normals",
    "bshot_query_normals", "bshot_set_normals", "bshot_compute_shot", "bshot_compute_lrf",
    "bshot_binarize", "bshot_compute_descriptors", "bshot_match", "bshot_match_mutual",
    "bshot_process_frame", "bshot_process_frame_dev", "bshot_fetch_frame", "bshot_ctx_enable_timing",
    "bshot_stage_times", "bshot_frame_counters", "bshot_map_reset", "bshot_map_append",
    "bshot_map_size", "bshot_match_shard_dev", "bshot_match_dev", "bshot_merge_cands_dev",
    "bshot_match_map", "bshot_reverse_owned_dev", "bshot_apply_rq_dev", "bshot_push_cands_dev",
    "bshot_reverse_owned_push_dev", "bshot_peer_barrier_dev", "bshot_peer_barrier_timeouts", "bshot_peer_barrier_reset", "bshot_launch_count", "bshot_popc_peak", "bshot_debug_counters", "bshot_map_append_dev", "bshot_comm_create", "bshot_comm_export", "bshot_comm_import",
    "bshot_comm_region", "bshot_comm_import_ptrs", "bshot_comm_destroy", "bshot_comm_check", "bshot_match_map_sharded_dev",
    "bshot_match_map_sharded", "bshot_gmap_create", "bshot_gmap_reset", "bshot_gmap_size", "bshot_gmap_add",
    "bshot_gmap_update_from_frame", "bshot_gmap_get_keypoints", "bshot_extract_frame", "bshot_match_frame_to_map", "bshot_frame_commit", "bshot_ransac",
    "bshot_preprocess", "bshot_preprocess_select", "bshot_extract_scan", "bshot_icp", "bshot_evaluate_estimation", "bshot_set_matcher",
    "bshot_iss_params_default", "bshot_detect_iss", "bshot_kp_repeatability", "bshot_voxel_grid",
    "bshot_odom_params_default", "bshot_odometry_step", "bshot_odometry_step_cloud", "bshot_odometry_reset", "bshot_ransac_dev",
    "bshot_gmap_export", "bshot_gmap_import", "bshot_relocalize", "bshot_relocalize_cloud",
    "bshot_gmap_scans", "bshot_loop_params_default", "bshot_detect_loop", "bshot_gmap_reanchor",
    "bshot_graph_params_default", "bshot_optimize_trajectory",
]


class Params(C.Structure):
    _fields_ = [("kp_radius", C.c_float), ("kp_max_nn", C.c_int), ("sr_type", C.c_int),
                ("top_k", C.c_int), ("normal_radius", C.c_float), ("normal_max_nn", C.c_int),
                ("normals_mode", C.c_int), ("shot_radius", C.c_float)]


class IssParams(C.Structure):
    _fields_ = [("salient_radius", C.c_float), ("non_max_radius", C.c_float), ("gamma_21", C.c_double),
                ("gamma_32", C.c_double), ("min_neighbors", C.c_int)]


class OdomParams(C.Structure):
    _fields_ = [("front", Params), ("vert_init_rad", C.c_double), ("lowpt_th", C.c_double), ("map_range", C.c_float),
                ("ransac_iterations", C.c_int), ("inlier_threshold", C.c_float), ("run_icp", C.c_int)]


class OdomReport(C.Structure):
    _fields_ = [("pose", C.c_float * 16), ("T_ransac", C.c_float * 16), ("n_points", C.c_size_t), ("n_targets", C.c_size_t),
                ("n_keypoints", C.c_int), ("n_pairs", C.c_int), ("n_inliers", C.c_int), ("ransac_iterations", C.c_int),
                ("icp_iterations", C.c_int), ("should_update_map", C.c_int), ("was_initial", C.c_int),
                ("h_diff_rad", C.c_float), ("t_diff_mm", C.c_float)]


class RelocReport(C.Structure):
    _fields_ = [("pose", C.c_float * 16), ("T_ransac", C.c_float * 16), ("n_points", C.c_size_t), ("n_map", C.c_size_t),
                ("n_icp_targets", C.c_size_t), ("n_keypoints", C.c_int), ("n_pairs", C.c_int), ("n_inliers", C.c_int),
                ("ransac_iterations", C.c_int), ("icp_iterations", C.c_int), ("accepted", C.c_int)]


class LoopParams(C.Structure):
    _fields_ = [("min_gap", C.c_int), ("min_inliers", C.c_int), ("ransac_iterations", C.c_int), ("inlier_threshold", C.c_float),
                ("map_range", C.c_float), ("run_icp", C.c_int)]


class GraphEdge(C.Structure):
    _fields_ = [("from_", C.c_int32), ("to", C.c_int32), ("T", C.c_float * 16)]


class GraphParams(C.Structure):
    _fields_ = [("odom_sigma_mm", C.c_float), ("odom_sigma_deg", C.c_float), ("loop_sigma_mm", C.c_float), ("loop_sigma_deg", C.c_float),
                ("max_iterations", C.c_int), ("max_cg_iterations", C.c_int), ("grad_tolerance", C.c_double), ("step_tolerance", C.c_double),
                ("cg_tolerance", C.c_double)]


class GraphReport(C.Structure):
    _fields_ = [("n_nodes", C.c_int), ("n_edges", C.c_int), ("iterations", C.c_int), ("cg_iterations", C.c_int), ("status", C.c_int),
                ("cost_initial", C.c_double), ("cost_final", C.c_double), ("grad_inf_final", C.c_double)]


class LoopReport(C.Structure):
    _fields_ = [("T_loop", C.c_float * 16), ("T_ransac", C.c_float * 16), ("T_rel", C.c_float * 16), ("pose", C.c_float * 16),
                ("n_candidates", C.c_size_t), ("n_icp_targets", C.c_size_t), ("scan", C.c_int), ("match_scan", C.c_int), ("votes", C.c_int),
                ("n_keypoints", C.c_int), ("n_pairs", C.c_int), ("n_inliers", C.c_int), ("ransac_iterations", C.c_int),
                ("icp_iterations", C.c_int), ("accepted", C.c_int)]


E_INVALID, E_CAPACITY, E_CUDA, E_STATE = -1, -2, -3, -4

CAND_DTYPE = np.dtype([("k1", "<u8"), ("k2", "<u8"), ("rq", "<u4"), ("pad", "<u4")])
NONE_KEY = np.uint64(0xFFFFFFFFFFFFFFFF)


class BshotError(RuntimeError):
    def __init__(self, msg, code=None):
        super().__init__(msg)
        self.code = code


def build(verbose=False):
    """Compile csrc/*.cu for sm_100a into libbshot_b200.so (nvcc cross-compiles without a GPU)."""
    out = None if verbose else subprocess.DEVNULL
    subprocess.check_call(["make", "-C", os.path.join(_HERE, "csrc"), "-j8"], stdout=out, stderr=out)
    return LIB_PATH


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise BshotError(f"{LIB_PATH} is missing: build it with `make -C b-shot-slam_b200/csrc` "
                             "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        vp, sz, ci, cf = C.c_void_p, C.c_size_t, C.c_int, C.c_float
        L.bshot_last_error.restype = C.c_char_p
        L.bshot_version.restype = ci
        L.bshot_params_default.argtypes = [C.POINTER(Params)]
        L.bshot_ctx_create.argtypes = [C.POINTER(vp), ci, sz, sz, sz]
        L.bshot_ctx_destroy.argtypes = [vp]
        L.bshot_ctx_destroy.restype = None
        L.bshot_ctx_stream.argtypes = [vp]
        L.bshot_ctx_stream.restype = vp
        L.bshot_ctx_sync.argtypes = [vp]
        L.bshot_ctx_reset.argtypes = [vp]
        L.bshot_set_cloud.argtypes = [vp, vp, sz, sz]
        L.bshot_detect_keypoints.argtypes = [vp, cf, ci, ci, ci, vp, vp, vp, vp]
        L.bshot_seg_ratio.argtypes = [vp, cf, ci, ci, vp]
        L.bshot_set_keypoints.argtypes = [vp, vp, sz, sz]
        L.bshot_compute_normals.argtypes = [vp, ci, cf, ci, vp]
        L.bshot_query_normals.argtypes = [vp, vp, sz, cf, ci, vp]
        L.bshot_set_normals.argtypes = [vp, vp, sz]
        L.bshot_compute_shot.argtypes = [vp, cf, vp, vp, vp, vp, vp]
        L.bshot_compute_lrf.argtypes = [vp, cf, vp, vp]
        L.bshot_binarize.argtypes = [vp, vp, sz, sz, vp]
        L.bshot_compute_descriptors.argtypes = [vp, C.POINTER(Params), vp]
        L.bshot_match.argtypes = [vp, vp, sz, vp, sz, vp, vp, vp, vp, vp]
        L.bshot_match_mutual.argtypes = [vp, vp, sz, vp, sz, vp, vp, vp]
        L.bshot_process_frame.argtypes = [vp, C.POINTER(Params), vp, sz, sz, vp, vp, vp, vp, vp]
        L.bshot_process_frame_dev.argtypes = [vp, C.POINTER(Params), vp, sz, sz]
        L.bshot_fetch_frame.argtypes = [vp, ci, vp, vp, vp, vp, vp]
        L.bshot_ctx_enable_timing.argtypes = [vp, ci]
        L.bshot_stage_times.argtypes = [vp, C.POINTER(C.c_float * 8)]
        L.bshot_frame_counters.argtypes = [vp, C.POINTER(C.c_ulonglong * 4)]
        L.bshot_map_reset.argtypes = [vp]
        L.bshot_map_append.argtypes = [vp, vp, sz]
        L.bshot_map_size.argtypes = [vp, C.POINTER(sz)]
        L.bshot_map_append_dev.argtypes = [vp, vp, sz]
        L.bshot_gmap_create.argtypes = [vp, sz, sz]
        L.bshot_gmap_reset.argtypes = [vp]
        L.bshot_gmap_size.argtypes = [vp, C.POINTER(sz), C.POINTER(sz)]
        L.bshot_gmap_add.argtypes = [vp, vp, vp, vp, sz, vp]
        L.bshot_gmap_update_from_frame.argtypes = [vp, vp]
        L.bshot_gmap_get_keypoints.argtypes = [vp, vp, cf, vp, vp, sz, C.POINTER(sz)]
        L.bshot_extract_frame.argtypes = [vp, C.POINTER(Params), vp, sz, sz, vp, vp, vp, vp, vp]
        L.bshot_match_frame_to_map.argtypes = [vp, vp, cf, vp, vp, vp, C.POINTER(sz), vp, sz]
        L.bshot_frame_commit.argtypes = [vp]
        L.bshot_ransac.argtypes = [vp, vp, sz, vp, sz, vp, sz, ci, cf, vp, vp, vp, vp]
        L.bshot_icp.argtypes = [vp, vp, sz, vp, sz, vp, ci, vp, vp, vp, vp]
        L.bshot_evaluate_estimation.argtypes = [vp, vp, vp, ci, vp, sz, vp, sz, ci, vp, vp, vp, vp, vp]
        L.bshot_preprocess_select.argtypes = [vp, vp, vp, vp, sz, vp, sz, C.c_double, C.c_double, vp, sz, ci, ci, vp, sz, C.POINTER(sz)]
        L.bshot_extract_scan.argtypes = [vp, C.POINTER(Params), vp, vp, vp, sz, vp, sz, C.c_double, C.c_double, vp, sz, C.POINTER(sz), vp, vp, vp, vp, vp]
        L.bshot_preprocess.argtypes = [vp, vp, vp, vp, sz, vp, sz, C.c_double, C.c_double, vp, sz, C.POINTER(sz)]
        L.bshot_comm_create.argtypes = [vp, ci, ci, sz]
        L.bshot_comm_export.argtypes = [vp, vp]
        L.bshot_comm_import.argtypes = [vp, vp]
        L.bshot_comm_region.argtypes = [vp, C.POINTER(vp), C.POINTER(sz)]
        L.bshot_comm_import_ptrs.argtypes = [vp, C.POINTER(vp)]
        L.bshot_comm_destroy.argtypes = [vp]
        L.bshot_comm_check.argtypes = [vp]
        L.bshot_match_map_sharded_dev.argtypes = [vp, vp, sz, C.c_uint64, vp]
        L.bshot_match_map_sharded.argtypes = [vp, vp, sz, C.c_uint64, vp]
        L.bshot_match_shard_dev.argtypes = [vp, vp, sz, C.c_uint64, ci, vp]
        L.bshot_match_dev.argtypes = [vp, vp, sz, vp, sz, C.c_uint64, ci, vp]
        L.bshot_merge_cands_dev.argtypes = [vp, vp, sz, sz, vp]
        L.bshot_match_map.argtypes = [vp, vp, sz, C.c_uint64, vp]
        L.bshot_reverse_owned_dev.argtypes = [vp, vp, sz, C.c_uint64, vp, vp]
        L.bshot_apply_rq_dev.argtypes = [vp, vp, vp, sz]
        L.bshot_push_cands_dev.argtypes = [vp, vp, sz, vp, ci, ci]
        L.bshot_peer_barrier_dev.argtypes = [vp, vp, ci, ci]
        L.bshot_peer_barrier_timeouts.argtypes = [vp, C.POINTER(C.c_uint)]
        L.bshot_peer_barrier_reset.argtypes = [vp]
        L.bshot_reverse_owned_push_dev.argtypes = [vp, vp, sz, C.c_uint64, vp, vp, ci, ci]
        L.bshot_launch_count.argtypes = [vp]
        L.bshot_launch_count.restype = C.c_ulonglong
        L.bshot_popc_peak.argtypes = [vp, C.POINTER(C.c_double)]
        L.bshot_set_matcher.argtypes = [vp, ci]
        L.bshot_debug_counters.argtypes = [vp, C.POINTER(C.c_ulonglong * 8)]
        L.bshot_iss_params_default.argtypes = [C.POINTER(IssParams)]
        L.bshot_iss_params_default.restype = None
        L.bshot_detect_iss.argtypes = [vp, C.POINTER(IssParams), vp, vp, sz, C.POINTER(sz), vp]
        L.bshot_kp_repeatability.argtypes = [vp, vp, sz, vp, vp, sz, vp, cf, vp, vp, C.POINTER(sz)]
        L.bshot_voxel_grid.argtypes = [vp, vp, sz, sz, cf, cf, cf, vp, sz, C.POINTER(sz)]
        L.bshot_odom_params_default.argtypes = [C.POINTER(OdomParams)]
        L.bshot_odom_params_default.restype = None
        L.bshot_odometry_step.argtypes = [vp, C.POINTER(OdomParams), vp, vp, vp, sz, vp, sz, C.POINTER(OdomReport)]
        L.bshot_odometry_step_cloud.argtypes = [vp, C.POINTER(OdomParams), vp, sz, sz, C.POINTER(OdomReport)]
        L.bshot_odometry_reset.argtypes = [vp]
        L.bshot_ransac_dev.argtypes = [vp, vp, vp, vp, vp, sz, ci, cf, vp, vp, vp, vp]
        L.bshot_gmap_export.argtypes = [vp, vp, vp, sz, C.POINTER(sz)]
        L.bshot_gmap_import.argtypes = [vp, vp, vp, sz]
        L.bshot_relocalize.argtypes = [vp, C.POINTER(OdomParams), ci, vp, vp, vp, sz, vp, sz, C.POINTER(RelocReport)]
        L.bshot_relocalize_cloud.argtypes = [vp, C.POINTER(OdomParams), ci, vp, sz, sz, C.POINTER(RelocReport)]
        L.bshot_gmap_scans.argtypes = [vp, vp, sz, vp, sz, C.POINTER(sz), C.POINTER(sz)]
        L.bshot_loop_params_default.argtypes = [C.POINTER(LoopParams)]
        L.bshot_loop_params_default.restype = None
        L.bshot_detect_loop.argtypes = [vp, C.POINTER(LoopParams), C.POINTER(LoopReport)]
        L.bshot_gmap_reanchor.argtypes = [vp, vp, sz, vp]
        L.bshot_graph_params_default.argtypes = [C.POINTER(GraphParams)]
        L.bshot_graph_params_default.restype = None
        L.bshot_optimize_trajectory.argtypes = [vp, vp, sz, C.POINTER(GraphParams), vp, sz, vp, C.POINTER(GraphReport)]
        _LIB = L
    return _LIB


def _chk(rc):
    if rc != 0:
        raise BshotError(f"bshot error {rc}: {lib().bshot_last_error().decode()}", rc)


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def default_params(**kw):
    p = Params()
    lib().bshot_params_default(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise AttributeError(k)
        setattr(p, k, v)
    return p


def iss_default_params(**kw):
    """ISS parameters of issKpDetection (src/lidar_odometry.cpp:447-461); keyword arguments override fields"""
    p = IssParams()
    lib().bshot_iss_params_default(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise AttributeError(k)
        setattr(p, k, v)
    return p


def odom_default_params(**kw):
    """parameters of the odometry step (test/odometry_test.cpp:32-33, src/lidar_odometry.cpp:6,198,255,258); keyword
    arguments override fields, and the extraction fields (kp_radius, top_k, ...) reach `front`"""
    p = OdomParams()
    lib().bshot_odom_params_default(C.byref(p))
    for k, v in kw.items():
        if hasattr(p, k):
            setattr(p, k, v)
        elif hasattr(p.front, k):
            setattr(p.front, k, v)
        else:
            raise AttributeError(k)
    return p


def graph_params_default(**kw):
    """parameters of bshot_optimize_trajectory; keyword arguments override fields"""
    p = GraphParams()
    lib().bshot_graph_params_default(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise AttributeError(k)
        setattr(p, k, v)
    return p


def loop_params_default(**kw):
    """parameters of bshot_detect_loop; keyword arguments override fields"""
    p = LoopParams()
    lib().bshot_loop_params_default(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise AttributeError(k)
        setattr(p, k, v)
    return p


def _report(r):
    mats = [name for name, _ in type(r)._fields_ if name in ("pose", "T_ransac", "T_loop", "T_rel")]
    out = {name: getattr(r, name) for name, _ in type(r)._fields_ if name not in mats}
    for name in mats:
        out[name] = np.ctypeslib.as_array(getattr(r, name)).reshape(4, 4).copy()
    return out


def _pose12(pose):
    """None, a row-major [R|T] (12 values) or a 4 x 4 matrix -> 12 contiguous float32 (None stays None)"""
    if pose is None:
        return None
    m = np.asarray(pose, dtype=np.float32)
    if m.size == 16:
        m = m.reshape(4, 4)[:3]
    return np.ascontiguousarray(m.reshape(12))


def unpack_cands(cand):
    """structured candidate records -> dict of int arrays (idx/dist, -1 = none)"""
    k1, k2 = cand["k1"], cand["k2"]
    h1, h2 = k1 != NONE_KEY, k2 != NONE_KEY
    out = dict(
        idx1=np.where(h1, (k1 & np.uint64(0xFFFFFFFF)).astype(np.int64), -1),
        dist1=np.where(h1, (k1 >> np.uint64(32)).astype(np.int64), -1),
        idx2=np.where(h2, (k2 & np.uint64(0xFFFFFFFF)).astype(np.int64), -1),
        dist2=np.where(h2, (k2 >> np.uint64(32)).astype(np.int64), -1),
        rq=np.where(cand["rq"] != 0xFFFFFFFF, cand["rq"].astype(np.int64), -1))
    return out


class Context:
    """One bshot_ctx: device buffers + one stream (mirrors the `bshot cb` member of LidarOdometry,
    include/lidar_odometry.h:57)."""

    def __init__(self, device=0, max_points=131072, max_keypoints=16384, max_targets=0):
        h = C.c_void_p()
        _chk(lib().bshot_ctx_create(C.byref(h), device, max_points, max_keypoints, max_targets))
        self.h = h
        self.max_points, self.max_keypoints = max_points, max_keypoints
        self.n_points = 0
        self.n_kp = 0

    def close(self):
        if getattr(self, "h", None):
            lib().bshot_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def stream(self):
        return lib().bshot_ctx_stream(self.h)

    def sync(self):
        _chk(lib().bshot_ctx_sync(self.h))

    def reset(self):
        _chk(lib().bshot_ctx_reset(self.h))

    def launch_count(self):
        return int(lib().bshot_launch_count(self.h))

    def set_matcher(self, kind):
        """-1 by problem size (default), 0 XOR + POPC, 1 tensor cores, 2 / 3 pipelined tensor-core kernel"""
        _chk(lib().bshot_set_matcher(self.h, int(kind)))

    def popc_peak(self):
        v = C.c_double()
        _chk(lib().bshot_popc_peak(self.h, C.byref(v)))
        return v.value

    # a1
    def set_cloud(self, xyz):
        xyz = np.ascontiguousarray(xyz, dtype=np.float32)
        assert xyz.ndim == 2 and xyz.shape[1] in (3, 4)
        _chk(lib().bshot_set_cloud(self.h, _p(xyz), xyz.shape[0], xyz.shape[1] * 4))
        self.n_points = xyz.shape[0]

    # a2 / a3
    def seg_ratio(self, radius=3000.0, max_nn=300, sr_type=SR_CV):
        out = np.empty(self.n_points, np.float32)
        _chk(lib().bshot_seg_ratio(self.h, radius, max_nn, sr_type, _p(out)))
        return out

    def detect_keypoints(self, radius=3000.0, max_nn=300, sr_type=SR_CV, top_k=600):
        idx = np.empty(top_k, np.int32)
        ratio = np.empty(top_k, np.float32)
        xyz = np.empty((top_k, 3), np.float32)
        cnt = C.c_int()
        _chk(lib().bshot_detect_keypoints(self.h, radius, max_nn, sr_type, top_k, _p(idx), _p(ratio),
                                          _p(xyz), C.byref(cnt)))
        k = cnt.value
        self.n_kp = k
        return idx[:k].copy(), ratio[:k].copy(), xyz[:k].copy()

    def set_keypoints(self, kp):
        kp = np.ascontiguousarray(kp, dtype=np.float32).reshape(-1, 3)
        _chk(lib().bshot_set_keypoints(self.h, _p(kp), kp.shape[0], 12))
        self.n_kp = kp.shape[0]

    # a4
    def compute_normals(self, mode=NORMALS_REFERENCE, radius=3000.0, max_nn=300):
        out = np.empty((self.n_points, 4), np.float32)
        _chk(lib().bshot_compute_normals(self.h, mode, radius, max_nn, _p(out)))
        return out

    def query_normals(self, q, radius=3000.0, max_nn=300):
        q = np.ascontiguousarray(q, dtype=np.float32).reshape(-1, 3)
        out = np.empty((q.shape[0], 4), np.float32)
        _chk(lib().bshot_query_normals(self.h, _p(q), q.shape[0], radius, max_nn, _p(out)))
        return out

    def set_normals(self, normals4):
        normals4 = np.ascontiguousarray(normals4, dtype=np.float32).reshape(-1, 4)
        _chk(lib().bshot_set_normals(self.h, _p(normals4), normals4.shape[0]))

    # a5..a7
    def compute_lrf(self, radius=3000.0):
        rf = np.empty((self.n_kp, 9), np.float32)
        nn = np.empty(self.n_kp, np.int32)
        _chk(lib().bshot_compute_lrf(self.h, radius, _p(rf), _p(nn)))
        return rf, nn

    def compute_shot(self, radius=3000.0, want_shot=True):
        k = self.n_kp
        bits = np.empty((k, 6), np.uint64)
        shot = np.empty((k, 352), np.float32) if want_shot else None
        rf = np.empty((k, 9), np.float32)
        nn = np.empty(k, np.int32)
        tot = C.c_longlong()
        _chk(lib().bshot_compute_shot(self.h, radius, _p(bits), _p(shot), _p(rf), _p(nn), C.byref(tot)))
        return dict(bits=bits, shot=shot, rf=rf, nn=nn, sum_neighbours=tot.value)

    def binarize(self, shot, stride_floats=None):
        shot = np.ascontiguousarray(shot, dtype=np.float32)
        if stride_floats is None:
            shot = shot.reshape(-1, 352)
            stride_floats = 352
        k = shot.size // stride_floats
        bits = np.empty((k, 6), np.uint64)
        _chk(lib().bshot_binarize(self.h, _p(shot), k, stride_floats, _p(bits)))
        return bits

    def compute_descriptors(self, params=None):
        bits = np.empty((self.n_kp, 6), np.uint64)
        _chk(lib().bshot_compute_descriptors(self.h, C.byref(params) if params else None, _p(bits)))
        return bits

    # a10 / a11
    def match(self, q, t, want_right=True):
        q = np.ascontiguousarray(q, dtype=np.uint64).reshape(-1, 6)
        t = np.ascontiguousarray(t, dtype=np.uint64).reshape(-1, 6)
        nq, nt = q.shape[0], t.shape[0]
        li, ld, li2, ld2 = (np.empty(nq, np.int32) for _ in range(4))
        ri = np.empty(nt, np.int32) if want_right else None
        _chk(lib().bshot_match(self.h, _p(q), nq, _p(t), nt, _p(li), _p(ld), _p(li2), _p(ld2), _p(ri)))
        return dict(left_idx=li, left_dist=ld, left_idx2=li2, left_dist2=ld2, right_idx=ri)

    def match_mutual(self, q, t):
        q = np.ascontiguousarray(q, dtype=np.uint64).reshape(-1, 6)
        t = np.ascontiguousarray(t, dtype=np.uint64).reshape(-1, 6)
        nq = q.shape[0]
        pairs = np.empty((max(nq, 1), 2), np.int32)
        dist = np.empty(max(nq, 1), np.int32)
        cnt = C.c_int()
        _chk(lib().bshot_match_mutual(self.h, _p(q), nq, _p(t), t.shape[0], _p(pairs), _p(dist), C.byref(cnt)))
        return pairs[:cnt.value].copy(), dist[:cnt.value].copy()

    # whole frame
    def process_frame(self, xyz, params):
        xyz = np.ascontiguousarray(xyz, dtype=np.float32)
        k = params.top_k
        kp_idx = np.empty(k, np.int32)
        bits = np.empty((k, 6), np.uint64)
        pairs = np.empty((k, 2), np.int32)
        nk, npairs = C.c_int(), C.c_int()
        _chk(lib().bshot_process_frame(self.h, C.byref(params), _p(xyz), xyz.shape[0], xyz.shape[1] * 4,
                                       _p(kp_idx), _p(bits), C.byref(nk), _p(pairs), C.byref(npairs)))
        self.n_points = xyz.shape[0]
        self.n_kp = nk.value
        return dict(kp_idx=kp_idx[:nk.value].copy(), bits=bits[:nk.value].copy(),
                    pairs=pairs[:npairs.value].copy())

    def process_frame_raw(self, xyz_ptr, n, stride_bytes, params, kp_idx_ptr, bits_ptr, pairs_ptr):
        """pointer-level variant for bench.py (pinned host buffers, no numpy allocation)"""
        nk, npairs = C.c_int(), C.c_int()
        _chk(lib().bshot_process_frame(self.h, C.byref(params), xyz_ptr, n, stride_bytes, kp_idx_ptr,
                                       bits_ptr, C.byref(nk), pairs_ptr, C.byref(npairs)))
        return nk.value, npairs.value

    def process_frame_dev(self, d_xyz_ptr, n, stride_bytes, params):
        """device-resident cloud (raw device pointer), asynchronous on the context stream"""
        _chk(lib().bshot_process_frame_dev(self.h, C.byref(params), d_xyz_ptr, n, stride_bytes))
        self.n_points = n

    def fetch_frame(self, top_k):
        kp_idx = np.empty(top_k, np.int32)
        bits = np.empty((top_k, 6), np.uint64)
        pairs = np.empty((top_k, 2), np.int32)
        nk, npairs = C.c_int(), C.c_int()
        _chk(lib().bshot_fetch_frame(self.h, top_k, _p(kp_idx), _p(bits), C.byref(nk), _p(pairs), C.byref(npairs)))
        self.n_kp = nk.value
        return dict(kp_idx=kp_idx[:nk.value].copy(), bits=bits[:nk.value].copy(), pairs=pairs[:npairs.value].copy())

    def enable_timing(self, on=True):
        _chk(lib().bshot_ctx_enable_timing(self.h, int(on)))

    def stage_times(self):
        a = (C.c_float * 8)()
        _chk(lib().bshot_stage_times(self.h, C.byref(a)))
        names = ["voxel_build", "seg_ratio", "topk", "normals", "shot_bshot", "match", "frame"]
        return {k: float(a[i]) for i, k in enumerate(names)}

    def frame_counters(self):
        a = (C.c_ulonglong * 4)()
        _chk(lib().bshot_frame_counters(self.h, C.byref(a)))
        return dict(detector_neighbours=int(a[0]), normals_neighbours=int(a[1]), shot_neighbours=int(a[2]),
                    keypoints=int(a[3]))

    def debug_counters(self):
        a = (C.c_ulonglong * 8)()
        _chk(lib().bshot_debug_counters(self.h, C.byref(a)))
        names = ["detector_neighbours", "normals_neighbours", "tiles_staged", "tile_points_swept", "query_attempts",
                 "unresolved_attempts", "fallback_queries", "blocks"]
        return {k: int(a[i]) for i, k in enumerate(names)}

    # sharded map
    def map_reset(self):
        _chk(lib().bshot_map_reset(self.h))

    def map_append(self, desc):
        desc = np.ascontiguousarray(desc, dtype=np.uint64).reshape(-1, 6)
        _chk(lib().bshot_map_append(self.h, _p(desc), desc.shape[0]))

    def map_append_dev(self, d_desc_ptr, n):
        _chk(lib().bshot_map_append_dev(self.h, d_desc_ptr, n))

    # GPU-resident global map + frame-to-map flow
    def gmap_create(self, max_entries, max_blocks=4096):
        _chk(lib().bshot_gmap_create(self.h, max_entries, max_blocks))

    def gmap_reset(self):
        _chk(lib().bshot_gmap_reset(self.h))

    def gmap_size(self):
        n, d = C.c_size_t(), C.c_size_t()
        _chk(lib().bshot_gmap_size(self.h, C.byref(n), C.byref(d)))
        return n.value, d.value

    def gmap_add(self, xyz, ratio, desc, pose=None):
        xyz = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
        ratio = np.ascontiguousarray(ratio, dtype=np.float32).reshape(-1)
        desc = np.ascontiguousarray(desc, dtype=np.uint64).reshape(-1, 6)
        pose = None if pose is None else np.ascontiguousarray(pose, dtype=np.float32).reshape(12)
        _chk(lib().bshot_gmap_add(self.h, _p(xyz), _p(ratio), _p(desc), xyz.shape[0], _p(pose)))

    def gmap_update_from_frame(self, pose=None):
        pose = None if pose is None else np.ascontiguousarray(pose, dtype=np.float32).reshape(12)
        _chk(lib().bshot_gmap_update_from_frame(self.h, _p(pose)))

    def gmap_get_keypoints(self, pos, rng, cap=1 << 20):
        pos = np.ascontiguousarray(pos, dtype=np.float32).reshape(3)
        n = C.c_size_t()
        _chk(lib().bshot_gmap_get_keypoints(self.h, _p(pos), rng, None, None, 0, C.byref(n)))
        xyz = np.empty((n.value, 3), np.float32)
        desc = np.empty((n.value, 6), np.uint64)
        _chk(lib().bshot_gmap_get_keypoints(self.h, _p(pos), rng, _p(xyz), _p(desc), n.value, C.byref(n)))
        return xyz, desc

    def gmap_export(self):
        """every map entry in map order (blocks in ascending lattice coordinates, x outermost; entries of a block in
        insertion order) -> (xyzr (n, 4) float32 {x, y, z, seg_ratio}, desc (n, 6) uint64)"""
        n = C.c_size_t()
        rc = lib().bshot_gmap_export(self.h, None, None, 0, C.byref(n))
        if rc not in (0, E_CAPACITY):
            _chk(rc)
        xyzr = np.empty((n.value, 4), np.float32)
        desc = np.empty((n.value, 6), np.uint64)
        _chk(lib().bshot_gmap_export(self.h, _p(xyzr), _p(desc), n.value, C.byref(n)))
        return xyzr, desc

    def gmap_import(self, xyzr, desc):
        """replace the map by these entries (a gmap_export result restores its map); on an error the map is empty"""
        xyzr = np.ascontiguousarray(xyzr, dtype=np.float32).reshape(-1, 4)
        desc = np.ascontiguousarray(desc, dtype=np.uint64).reshape(-1, 6)
        if xyzr.shape[0] != desc.shape[0]:
            raise BshotError("gmap_import: xyzr and desc differ in length", E_INVALID)
        _chk(lib().bshot_gmap_import(self.h, _p(xyzr), _p(desc), xyzr.shape[0]))

    def gmap_scans(self):
        """the update that wrote each entry, in gmap_export's order, and the pose each update used ->
        (entry_scans (n,) uint32, poses (m, 4, 4) float32 row-major)"""
        n, m = C.c_size_t(), C.c_size_t()
        rc = lib().bshot_gmap_scans(self.h, None, 0, None, 0, C.byref(n), C.byref(m))
        if rc not in (0, E_CAPACITY):
            _chk(rc)
        tags = np.empty(n.value, np.uint32)
        p12 = np.empty((m.value, 3, 4), np.float32)
        _chk(lib().bshot_gmap_scans(self.h, _p(tags), n.value, _p(p12), m.value, C.byref(n), C.byref(m)))
        poses = np.zeros((m.value, 4, 4), np.float32)
        poses[:, :3] = p12
        poses[:, 3, 3] = 1.0
        return tags, poses

    def extract_frame(self, xyz, params):
        xyz = np.ascontiguousarray(xyz, dtype=np.float32)
        k = params.top_k
        idx, kp, ratio, bits = np.empty(k, np.int32), np.empty((k, 3), np.float32), np.empty(k, np.float32), np.empty((k, 6), np.uint64)
        nk = C.c_int()
        _chk(lib().bshot_extract_frame(self.h, C.byref(params), _p(xyz), xyz.shape[0], xyz.shape[1] * 4, _p(idx), _p(kp), _p(ratio),
                                       _p(bits), C.byref(nk)))
        n = nk.value
        self.n_points, self.n_kp = xyz.shape[0], n
        return dict(kp_idx=idx[:n].copy(), kp_xyz=kp[:n].copy(), seg_ratio=ratio[:n].copy(), bits=bits[:n].copy())

    def match_frame_to_map(self, ref_pos, rng=100000.0, ref_pose=None, target_cap=1 << 20):
        ref_pos = np.ascontiguousarray(ref_pos, dtype=np.float32).reshape(3)
        ref_pose = None if ref_pose is None else np.ascontiguousarray(ref_pose, dtype=np.float32).reshape(12)
        pairs = np.empty((max(self.max_keypoints, 1), 2), np.int32)
        npairs, nt = C.c_int(), C.c_size_t()
        txyz = np.empty((target_cap, 3), np.float32)
        _chk(lib().bshot_match_frame_to_map(self.h, _p(ref_pos), rng, _p(ref_pose), _p(pairs), C.byref(npairs), C.byref(nt), _p(txyz), target_cap))
        return dict(pairs=pairs[:npairs.value].copy(), n_targets=nt.value, target_xyz=txyz[:nt.value].copy())

    def ransac(self, src_xyz, tgt_xyz, pairs, max_iterations=2000, threshold=1500.0):
        src_xyz = np.ascontiguousarray(src_xyz, dtype=np.float32).reshape(-1, 3)
        tgt_xyz = np.ascontiguousarray(tgt_xyz, dtype=np.float32).reshape(-1, 3)
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        out = np.empty((max(len(pairs), 1), 2), np.int32)
        T = np.empty((4, 4), np.float32)
        n, it = C.c_int(), C.c_int()
        _chk(lib().bshot_ransac(self.h, _p(src_xyz), src_xyz.shape[0], _p(tgt_xyz), tgt_xyz.shape[0], _p(pairs), pairs.shape[0],
                                max_iterations, threshold, _p(out), C.byref(n), _p(T), C.byref(it)))
        return dict(pairs=out[:n.value].copy(), transform=T, iterations=it.value)

    def icp(self, src_xyz, tgt_xyz, pre=None, max_iterations=10):
        """pcl::IterativeClosestPoint with PCL's defaults (src/lidar_odometry.cpp:283-291) on src moved by `pre`"""
        src_xyz = np.ascontiguousarray(src_xyz, dtype=np.float32).reshape(-1, 3)
        tgt_xyz = np.ascontiguousarray(tgt_xyz, dtype=np.float32).reshape(-1, 3)
        pre = None if pre is None else np.ascontiguousarray(pre, dtype=np.float32).reshape(16)
        T = np.empty((4, 4), np.float32)
        it, st, mse = C.c_int(), C.c_int(), C.c_double()
        _chk(lib().bshot_icp(self.h, _p(src_xyz), src_xyz.shape[0], _p(tgt_xyz), tgt_xyz.shape[0], _p(pre), max_iterations, _p(T), C.byref(it),
                             C.byref(st), C.byref(mse)))
        return dict(transform=T, iterations=it.value, state=st.value, mse=mse.value)

    def evaluate_estimation(self, T_ransac, T_ref, n_corr, src_kp, tgt_kp, run_icp=True):
        """LidarOdometry::evaluateEstimation (src/lidar_odometry.cpp:267-296)"""
        T_ransac = np.ascontiguousarray(T_ransac, dtype=np.float32).reshape(16)
        T_ref = np.ascontiguousarray(T_ref, dtype=np.float32).reshape(16)
        src_kp = np.ascontiguousarray(src_kp, dtype=np.float32).reshape(-1, 3)
        tgt_kp = np.ascontiguousarray(tgt_kp, dtype=np.float32).reshape(-1, 3)
        T = np.empty((4, 4), np.float32)
        upd, it, h, t = C.c_int(), C.c_int(), C.c_float(), C.c_float()
        _chk(lib().bshot_evaluate_estimation(self.h, _p(T_ransac), _p(T_ref), n_corr, _p(src_kp), src_kp.shape[0], _p(tgt_kp), tgt_kp.shape[0],
                                             1 if run_icp else 0, _p(T), C.byref(upd), C.byref(h), C.byref(t), C.byref(it)))
        return dict(T_best=T, should_update_map=bool(upd.value), h_diff=h.value, t_diff=t.value, icp_iterations=it.value)

    def preprocess(self, azimuth_deg, vertical_deg, distance, ring_deg, vert_init=-0.6, lowpt_th=-1950.0, select=None, save_selected=True):
        """Preprocessor::run (src/preprocess.cpp:213-223) on one rotation of returns sorted by azimuth -> (m, 3) float32 mm."""
        az = np.ascontiguousarray(azimuth_deg, dtype=np.float64)
        ve = np.ascontiguousarray(vertical_deg, dtype=np.float64)
        di = np.ascontiguousarray(distance, dtype=np.uint16)
        ring = np.ascontiguousarray(ring_deg, dtype=np.float64)
        assert az.shape == ve.shape == di.shape
        out = np.empty((max(az.size, 1), 3), np.float32)
        n = C.c_size_t()
        sel = None if select is None else np.ascontiguousarray(select, dtype=np.int32)
        _chk(lib().bshot_preprocess_select(self.h, _p(az), _p(ve), _p(di), az.size, _p(ring), ring.size, vert_init, lowpt_th, _p(sel),
                                           0 if sel is None else sel.size, 0 if sel is None else 1, 1 if save_selected else 0, _p(out), out.shape[0], C.byref(n)))
        return out[:n.value].copy()

    def extract_scan(self, azimuth_deg, vertical_deg, distance, ring_deg, params, vert_init=-0.6, lowpt_th=-1950.0, want_cloud=True):
        """lasers -> preprocessed cloud (device resident) -> keypoints + descriptors in one call"""
        az = np.ascontiguousarray(azimuth_deg, dtype=np.float64)
        ve = np.ascontiguousarray(vertical_deg, dtype=np.float64)
        di = np.ascontiguousarray(distance, dtype=np.uint16)
        ring = np.ascontiguousarray(ring_deg, dtype=np.float64)
        k = params.top_k
        cloud = np.empty((max(az.size, 1), 3), np.float32) if want_cloud else None
        idx, kp, ratio, bits = np.empty(k, np.int32), np.empty((k, 3), np.float32), np.empty(k, np.float32), np.empty((k, 6), np.uint64)
        npts, nk = C.c_size_t(), C.c_int()
        _chk(lib().bshot_extract_scan(self.h, C.byref(params), _p(az), _p(ve), _p(di), az.size, _p(ring), ring.size, vert_init, lowpt_th, _p(cloud),
                                      0 if cloud is None else cloud.shape[0], C.byref(npts), _p(idx), _p(kp), _p(ratio), _p(bits), C.byref(nk)))
        n = nk.value
        self.n_points, self.n_kp = npts.value, n
        return dict(cloud=None if cloud is None else cloud[:npts.value].copy(), n_points=npts.value, kp_idx=idx[:n].copy(), kp_xyz=kp[:n].copy(),
                    seg_ratio=ratio[:n].copy(), bits=bits[:n].copy())

    def frame_commit(self):
        _chk(lib().bshot_frame_commit(self.h))

    # the per-scan odometry step (lasers or a preprocessed cloud -> pose in one call)
    def odometry_step(self, azimuth_deg, vertical_deg, distance, ring_deg, params=None):
        """Preprocessor::run -> extraction -> matching -> RANSAC -> gate + ICP -> pose -> map update -> reference frame, on
        the device.  Returns the report as a dict; "pose" (4 x 4 float32, row-major) is T_best.  Needs gmap_create first."""
        params = odom_default_params() if params is None else params
        az = np.ascontiguousarray(azimuth_deg, dtype=np.float64)
        ve = np.ascontiguousarray(vertical_deg, dtype=np.float64)
        di = np.ascontiguousarray(distance, dtype=np.uint16)
        ring = np.ascontiguousarray(ring_deg, dtype=np.float64)
        assert az.shape == ve.shape == di.shape
        r = OdomReport()
        _chk(lib().bshot_odometry_step(self.h, C.byref(params), _p(az), _p(ve), _p(di), az.size, _p(ring), ring.size, C.byref(r)))
        self.n_points, self.n_kp = r.n_points, r.n_keypoints
        return _report(r)

    def odometry_step_cloud(self, xyz, params=None):
        """the same on an already-preprocessed (N, 3) or (N, 4) float32 cloud"""
        params = odom_default_params() if params is None else params
        xyz = np.ascontiguousarray(xyz, dtype=np.float32)
        assert xyz.ndim == 2 and xyz.shape[1] in (3, 4)
        r = OdomReport()
        _chk(lib().bshot_odometry_step_cloud(self.h, C.byref(params), _p(xyz), xyz.shape[0], xyz.shape[1] * 4, C.byref(r)))
        self.n_points, self.n_kp = r.n_points, r.n_keypoints
        return _report(r)

    def relocalize(self, azimuth_deg, vertical_deg, distance, ring_deg, params=None, min_inliers=15):
        """one rotation against the whole map without a prior pose: extraction -> matching against every map entry ->
        RANSAC -> ICP around T_ransac.  With n_inliers >= min_inliers the pose becomes "pose" (T_best), the status RUN, and
        the map and reference frame move on as after a step; otherwise nothing changes.  Returns the report as a dict."""
        params = odom_default_params() if params is None else params
        az = np.ascontiguousarray(azimuth_deg, dtype=np.float64)
        ve = np.ascontiguousarray(vertical_deg, dtype=np.float64)
        di = np.ascontiguousarray(distance, dtype=np.uint16)
        ring = np.ascontiguousarray(ring_deg, dtype=np.float64)
        assert az.shape == ve.shape == di.shape
        r = RelocReport()
        _chk(lib().bshot_relocalize(self.h, C.byref(params), min_inliers, _p(az), _p(ve), _p(di), az.size, _p(ring), ring.size, C.byref(r)))
        self.n_points, self.n_kp = r.n_points, r.n_keypoints
        return _report(r)

    def relocalize_cloud(self, xyz, params=None, min_inliers=15):
        """the same on an already-preprocessed (N, 3) or (N, 4) float32 cloud"""
        params = odom_default_params() if params is None else params
        xyz = np.ascontiguousarray(xyz, dtype=np.float32)
        assert xyz.ndim == 2 and xyz.shape[1] in (3, 4)
        r = RelocReport()
        _chk(lib().bshot_relocalize_cloud(self.h, C.byref(params), min_inliers, _p(xyz), xyz.shape[0], xyz.shape[1] * 4, C.byref(r)))
        self.n_points, self.n_kp = r.n_points, r.n_keypoints
        return _report(r)

    def detect_loop(self, params=None):
        """is the last scan the odometry took a revisit of a scan at least params.min_gap updates older?  Read only.
        Returns the report as a dict: T_loop / T_ransac / T_rel / pose (4 x 4 float32), match_scan, votes, accepted, ..."""
        params = loop_params_default() if params is None else params
        r = LoopReport()
        _chk(lib().bshot_detect_loop(self.h, C.byref(params), C.byref(r)))
        return _report(r)

    def gmap_reanchor(self, poses):
        """move the map to a corrected trajectory: poses (n, 4, 4) or (n, 3, 4), the corrected pose of every map update
        (n = len(gmap_scans()[1])).  Each entry moves by T'_u * T_u^-1 of the update u that wrote it; the trajectory
        becomes poses.  Returns the odometry's new pose (4 x 4 float32)"""
        p = np.asarray(poses, dtype=np.float32)
        if p.ndim != 3 or p.shape[1:] not in ((4, 4), (3, 4)):
            raise BshotError("gmap_reanchor: poses of shape (n, 4, 4) or (n, 3, 4) expected", E_INVALID)
        p12 = np.ascontiguousarray(p[:, :3, :])
        pose = np.empty((4, 4), np.float32)
        _chk(lib().bshot_gmap_reanchor(self.h, _p(p12), p12.shape[0], _p(pose)))
        return pose

    def optimize_trajectory(self, loops, params=None):
        """the trajectory's pose graph with these loop edges, optimised on the device (read only).  loops: detect_loop
        report dicts (edge (match_scan, scan), measurement T_rel) or (from, to, T 4 x 4) tuples.  Returns a dict: poses
        (n, 4, 4) float32, loop_cost (L,) float64 and the report fields"""
        params = graph_params_default() if params is None else params
        edges = (GraphEdge * max(len(loops), 1))()
        for k, e in enumerate(loops):
            if isinstance(e, dict):
                f, t, T = e["match_scan"], e["scan"], e["T_rel"]
            else:
                f, t, T = e
            edges[k].from_, edges[k].to = int(f), int(t)
            edges[k].T[:] = [float(v) for v in np.asarray(T, np.float32).reshape(16)]
        n = len(self.gmap_scans_poses())
        p12 = np.empty((max(n, 1), 3, 4), np.float32)
        cost = np.empty(max(len(loops), 1), np.float64)
        r = GraphReport()
        _chk(lib().bshot_optimize_trajectory(self.h, C.cast(edges, C.c_void_p), len(loops), C.byref(params), _p(p12), n, _p(cost), C.byref(r)))
        poses = np.zeros((n, 4, 4), np.float32)
        poses[:, :3] = p12[:n]
        poses[:, 3, 3] = 1.0
        out = {name: getattr(r, name) for name, _ in GraphReport._fields_}
        out.update(poses=poses, loop_cost=cost[:len(loops)].copy())
        return out

    def gmap_scans_poses(self):
        """the trajectory alone (no map gather) -> (m, 4, 4) float32"""
        m = C.c_size_t()
        _chk(lib().bshot_gmap_scans(self.h, None, 0, None, 0, None, C.byref(m)))
        p12 = np.empty((m.value, 3, 4), np.float32)
        _chk(lib().bshot_gmap_scans(self.h, None, 0, _p(p12), m.value, None, C.byref(m)))
        poses = np.zeros((m.value, 4, 4), np.float32)
        poses[:, :3] = p12
        poses[:, 3, 3] = 1.0
        return poses

    def odometry_reset(self):
        """INITIAL status, identity pose, empty map, no reference frame"""
        _chk(lib().bshot_odometry_reset(self.h))

    def ransac_dev(self, src4, tgt4, pairs, n_pairs, max_iterations=2000, threshold=1500.0):
        """bshot_ransac on CUDA tensors: src4 / tgt4 (N, 4) float32, pairs (P, 2) int32, n_pairs (1,) int32 (the valid
        prefix of pairs).  Returns dict(pairs, n_inliers, transform, iterations) of CUDA tensors; the call is complete
        on return."""
        import torch
        for t, dt in ((src4, torch.float32), (tgt4, torch.float32), (pairs, torch.int32), (n_pairs, torch.int32)):
            if not (t.is_cuda and t.dtype == dt and t.is_contiguous()):
                raise BshotError("ransac_dev: contiguous CUDA tensors of float32 (points) and int32 (pairs, count) expected", E_INVALID)
        cap = pairs.shape[0]
        dev = pairs.device
        out_pairs = torch.zeros((max(cap, 1), 2), dtype=torch.int32, device=dev)
        n_out = torch.zeros(1, dtype=torch.int32, device=dev)
        T = torch.zeros((4, 4), dtype=torch.float32, device=dev)
        it = torch.zeros(1, dtype=torch.int32, device=dev)
        torch.cuda.synchronize(dev)   # the inputs are complete before the context's stream reads them
        _chk(lib().bshot_ransac_dev(self.h, src4.data_ptr(), tgt4.data_ptr(), pairs.data_ptr(), n_pairs.data_ptr(), cap, max_iterations, threshold,
                                    out_pairs.data_ptr(), n_out.data_ptr(), T.data_ptr(), it.data_ptr()))
        self.sync()
        return dict(pairs=out_pairs, n_inliers=n_out, transform=T, iterations=it)

    # ISS keypoints + repeatability (the reference's kp_test evaluation)
    def detect_iss(self, params=None, want_eigs=False):
        """ISS keypoints of the cloud the context holds: dict(idx, xyz) in ascending point index, plus eigs (N x 3,
        lambda1..3) when want_eigs"""
        params = iss_default_params() if params is None else params
        cap = min(self.n_points, 8192)
        cnt = C.c_size_t()
        eigs = np.empty((self.n_points, 3), np.float64) if want_eigs else None
        while True:
            idx = np.empty(max(cap, 1), np.int32)
            xyz = np.empty((max(cap, 1), 3), np.float32)
            rc = lib().bshot_detect_iss(self.h, C.byref(params), _p(idx), _p(xyz), cap, C.byref(cnt), _p(eigs))
            if rc == E_CAPACITY and cnt.value > cap:
                cap = cnt.value
                continue
            _chk(rc)
            break
        k = cnt.value
        out = dict(idx=idx[:k].copy(), xyz=xyz[:k].copy())
        if want_eigs:
            out["eigs"] = eigs
        return out

    def kp_repeatability(self, a, b, pose_a=None, pose_b=None, radius=30.0):
        """nearest point of B for every point of A (both moved by their 3x4 poses): dict(nn_idx, nn_dist, hits, rate)"""
        a = np.ascontiguousarray(a, dtype=np.float32).reshape(-1, 3)
        b = np.ascontiguousarray(b, dtype=np.float32).reshape(-1, 3)
        pa, pb = _pose12(pose_a), _pose12(pose_b)
        na = a.shape[0]
        idx = np.empty(max(na, 1), np.int32)
        dist = np.empty(max(na, 1), np.float32)
        hits = C.c_size_t()
        _chk(lib().bshot_kp_repeatability(self.h, _p(a), na, _p(pa), _p(b), b.shape[0], _p(pb), radius, _p(idx), _p(dist), C.byref(hits)))
        return dict(nn_idx=idx[:na].copy(), nn_dist=dist[:na].copy(), hits=hits.value, rate=hits.value / na if na else 0.0)

    # voxel-grid downsampling (the reference's bshot::calculate_voxel_grid_keypoints)
    def voxel_grid(self, xyz, leaf):
        """pcl::VoxelGrid centroids of a host cloud ((N, 3) or (N, 4) float32; not the context's cloud, which stays as it
        was) with leaf sizes `leaf` (a scalar or a 3-sequence, mm) -> (M, 3) float32 in ascending voxel index"""
        xyz = np.ascontiguousarray(xyz, dtype=np.float32)
        assert xyz.ndim == 2 and xyz.shape[1] in (3, 4)
        lx, ly, lz = (float(v) for v in np.broadcast_to(np.asarray(leaf, dtype=np.float32), (3,)))
        cap = min(xyz.shape[0], 16384)
        cnt = C.c_size_t()
        while True:
            out = np.empty((max(cap, 1), 3), np.float32)
            rc = lib().bshot_voxel_grid(self.h, _p(xyz), xyz.shape[0], xyz.shape[1] * 4, lx, ly, lz, _p(out), cap, C.byref(cnt))
            if rc == E_CAPACITY and cnt.value > cap:
                cap = cnt.value
                continue
            _chk(rc)
            break
        return out[:cnt.value].copy()

    # multi-rank exchange behind the C ABI (CUDA IPC peer memory)
    def comm_create(self, rank, nranks, max_queries):
        _chk(lib().bshot_comm_create(self.h, rank, nranks, max_queries))

    def comm_export(self):
        h = np.zeros(64, np.uint8)
        _chk(lib().bshot_comm_export(self.h, _p(h)))
        return h

    def comm_import(self, handles):
        handles = np.ascontiguousarray(handles, dtype=np.uint8).reshape(-1, 64)
        _chk(lib().bshot_comm_import(self.h, _p(handles)))

    def comm_region(self):
        ptr, n = C.c_void_p(), C.c_size_t()
        _chk(lib().bshot_comm_region(self.h, C.byref(ptr), C.byref(n)))
        return ptr.value, n.value

    def comm_import_ptrs(self, ptrs):
        arr = (C.c_void_p * len(ptrs))(*[C.c_void_p(p) for p in ptrs])
        _chk(lib().bshot_comm_import_ptrs(self.h, arr))

    def comm_destroy(self):
        _chk(lib().bshot_comm_destroy(self.h))

    def comm_check(self):
        _chk(lib().bshot_comm_check(self.h))

    def match_map_sharded_dev(self, d_q_ptr, nq, global_base, d_cand_ptr):
        _chk(lib().bshot_match_map_sharded_dev(self.h, d_q_ptr, nq, global_base, d_cand_ptr))

    def match_map_sharded(self, q, global_base=0):
        q = np.ascontiguousarray(q, dtype=np.uint64).reshape(-1, 6)
        cand = np.empty(q.shape[0], CAND_DTYPE)
        _chk(lib().bshot_match_map_sharded(self.h, _p(q), q.shape[0], global_base, _p(cand)))
        return cand

    def map_size(self):
        n = C.c_size_t()
        _chk(lib().bshot_map_size(self.h, C.byref(n)))
        return n.value

    def match_map(self, q, global_base=0):
        q = np.ascontiguousarray(q, dtype=np.uint64).reshape(-1, 6)
        cand = np.empty(q.shape[0], CAND_DTYPE)
        _chk(lib().bshot_match_map(self.h, _p(q), q.shape[0], global_base, _p(cand)))
        return cand

    def match_shard_dev(self, d_q_ptr, nq, global_base, with_rq, d_cand_ptr):
        _chk(lib().bshot_match_shard_dev(self.h, d_q_ptr, nq, global_base, int(with_rq), d_cand_ptr))

    def match_dev(self, d_q_ptr, nq, d_t_ptr, nt, global_base, with_rq, d_cand_ptr):
        _chk(lib().bshot_match_dev(self.h, d_q_ptr, nq, d_t_ptr, nt, global_base, int(with_rq), d_cand_ptr))

    def reverse_owned_dev(self, d_q_ptr, nq, global_base, d_merged_ptr, d_rq_ptr):
        _chk(lib().bshot_reverse_owned_dev(self.h, d_q_ptr, nq, global_base, d_merged_ptr, d_rq_ptr))

    def apply_rq_dev(self, d_cands_ptr, d_rq_ptr, nq):
        _chk(lib().bshot_apply_rq_dev(self.h, d_cands_ptr, d_rq_ptr, nq))

    # peer-memory exchange (symmetric buffers): stores into every rank's buffers, the caller adds the barriers
    def push_cands_dev(self, d_cands_ptr, nq, d_peer_ptrs, nranks, rank):
        _chk(lib().bshot_push_cands_dev(self.h, d_cands_ptr, nq, d_peer_ptrs, nranks, rank))

    def peer_barrier_dev(self, d_peer_flag_ptrs, nranks, rank):
        _chk(lib().bshot_peer_barrier_dev(self.h, d_peer_flag_ptrs, nranks, rank))

    def peer_barrier_reset(self):
        _chk(lib().bshot_peer_barrier_reset(self.h))

    def peer_barrier_timeouts(self):
        e = C.c_uint()
        _chk(lib().bshot_peer_barrier_timeouts(self.h, C.byref(e)))
        return int(e.value)

    def reverse_owned_push_dev(self, d_q_ptr, nq, global_base, d_merged_ptr, d_peer_rq_ptrs, nranks, rank):
        _chk(lib().bshot_reverse_owned_push_dev(self.h, d_q_ptr, nq, global_base, d_merged_ptr, d_peer_rq_ptrs, nranks, rank))

    def merge_cands_dev(self, d_cands_ptr, nranks, nq, d_out_ptr):
        _chk(lib().bshot_merge_cands_dev(self.h, d_cands_ptr, nranks, nq, d_out_ptr))
