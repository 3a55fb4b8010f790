"""Pins the oracle and the CUDA path to REFERENCE-COMPILED code: oracle/_ref/libbshot_ref.so is the reference's
include/bshot_bits.h compiled unchanged (oracle/ref_shim.cpp; PCL names -> oracle/pcl_stub).
 * golden vectors produced by that library (tests/golden/ref_pin.npz, made by tests/golden/make_ref_pin.py) are
   checked on every machine, CPU (oracle) and GPU (-m gpu, through the C ABI);
 * larger random cases are compared live with that library where it is built, and everywhere with a regression
   snapshot of the oracle's output (tests/golden/snapshots.py); minVect is checked where the library is built.
Pinned outright (reference arithmetic end to end): compute_bshot_from_SHOT (include/bshot_bits.h:144-278), minVect
(:6-20) and the std::bitset<352> record.  Pinned as control flow + data placement around the oracle's PCL
restatement: calculate_normals (:43-94, keypoint-ordinal placement, persistent cloud1_normals) and calculate_SHOT."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
from snapshots import Snapshots  # noqa: E402


@pytest.fixture(scope="module")
def pin():
    return np.load(os.path.join(HERE, "golden", "ref_pin.npz"))


@pytest.fixture(scope="module")
def ref(oracle):
    if oracle.ref_lib() is None:
        pytest.skip("oracle/_ref/libbshot_ref.so not built (needs the reference sources at build time)")
    return oracle


class ExpectedReference:
    """expected output of bshot::compute_bshot_from_SHOT and of the featureMatching loops: snapshot of the oracle's output,
    plus the reference-compiled library's (oracle/_ref) where it is built"""

    def __init__(self, snapshots, oracle):
        self.snapshots, self.oracle = snapshots, oracle
        self.built = oracle.ref_lib() is not None

    def _oracle_matching(self, q, t):
        m = self.oracle.match(q, t)
        return dict(left_idx=m["left_idx"], right_idx=m["right_idx"], pairs=self.oracle.mutual(m["left_idx"], m["right_idx"]))

    def bshot(self, shot):
        return self.snapshots.expect("bshot_from_shot", (np.ascontiguousarray(shot, dtype=np.float32),), self.oracle.bshot, "oracle",
                                     self.oracle.ref_bshot if self.built else None)

    def feature_matching(self, q, t):
        args = (np.ascontiguousarray(q, dtype=np.uint64), np.ascontiguousarray(t, dtype=np.uint64))
        return self.snapshots.expect("feature_matching", args, self._oracle_matching, "oracle",
                                     self.oracle.ref_feature_matching if self.built else None)


@pytest.fixture(scope="module")
def expected(oracle):
    snapshots = Snapshots()
    yield ExpectedReference(snapshots, oracle)
    snapshots.save()


def flow_frames(synth, pin):
    s = int(pin["flow_stride"])
    return synth.make_scan("hdl32e", 0)[::s].copy(), synth.make_scan("hdl32e", 1)[::s].copy()


# ---- oracle vs reference-made golden vectors (any machine) -------------------------------------------------
def test_orc_bshot_matches_reference_vectors(oracle, pin):
    assert np.array_equal(oracle.bshot(pin["shot"]), pin["shot_bits"])


def test_orc_match_matches_reference_vectors(oracle, pin):
    m = oracle.match(pin["match_q"], pin["match_t"])
    assert np.array_equal(m["left_idx"], pin["match_left"])
    assert np.array_equal(m["right_idx"], pin["match_right"])
    assert np.array_equal(oracle.mutual(m["left_idx"], m["right_idx"]), pin["match_pairs"])


def test_orc_descriptor_flow_matches_reference_vectors(oracle, synth, pin):
    f0, f1 = flow_frames(synth, pin)
    d0 = oracle.Cloud(f0).compute_descriptors(pin["flow_kp0"], 3000.0, 300, oracle.MODE_REFERENCE, want_normals=True)
    assert np.array_equal(d0["bits"], pin["flow_bits0"])
    assert np.array_equal(d0["normals"][:128], pin["flow_normals0_head"], equal_nan=True)
    assert np.array_equal(d0["rf"], pin["flow_rf0"], equal_nan=True)
    assert np.array_equal(d0["shot"][:16], pin["flow_shot0"], equal_nan=True)
    # frame 1 has FEWER keypoints (64 < 96): the reference's persistent cloud1_normals keeps frame 0's keypoint
    # normals at indices [64, 96) (include/bshot_bits.h:59 resize keeps the prefix) -- rebuilt here by hand
    c1 = oracle.Cloud(f1)
    kn = c1.normals(pin["flow_kp1"], 3000.0, 300)
    normals = np.zeros((len(f1), 4), np.float32)
    normals[:96] = pin["flow_normals0_head"][:96]
    normals[:64] = kn
    assert np.array_equal(normals[:128], pin["flow_normals1_head"], equal_nan=True)
    shot, _, _, _ = c1.shot(pin["flow_kp1"], normals, 3000.0)
    assert np.array_equal(oracle.bshot(shot), pin["flow_bits1"])


# ---- live comparison with the reference-compiled library where it is built, snapshots everywhere -------------
def test_live_bshot_random(oracle, expected):
    rng = np.random.default_rng(5)
    s = (rng.random((4000, 352)) ** 8).astype(np.float32)
    s[rng.random(s.shape) < 0.6] = 0
    s[rng.random(s.shape) < 0.001] = np.nan
    expected.bshot(s).check(oracle.bshot(s), "B-SHOT bits")


def test_live_minvect_first_minimum(ref):
    assert ref.ref_minvect([5, 3, 3, 7, 3]) == (3, 1)
    assert ref.ref_minvect([0]) == (0, 0)
    assert ref.ref_minvect([9, 9, 9]) == (9, 0)


@pytest.mark.parametrize("nq,nt,seed", [(1, 1, 0), (7, 300, 1), (300, 7, 2), (257, 511, 3)])
def test_live_feature_matching(oracle, expected, synth, nq, nt, seed):
    q = synth.random_descriptors(nq, seed=100 + seed, density=30)
    t = synth.random_descriptors(nt, seed=200 + seed, density=30)
    t[nt // 2:] = t[: nt - nt // 2]                     # duplicated targets: ties everywhere
    r = expected.feature_matching(q, t)
    m = oracle.match(q, t)
    r["left_idx"].check(m["left_idx"], "left_idx")
    r["right_idx"].check(m["right_idx"], "right_idx")
    r["pairs"].check(oracle.mutual(m["left_idx"], m["right_idx"]), "pairs")


# ---- the CUDA path vs the same reference-made vectors --------------------------------------------------------
@pytest.mark.gpu
def test_gpu_binarize_matches_reference_vectors(gpu_ctx, pin):
    assert np.array_equal(gpu_ctx.binarize(pin["shot"]), pin["shot_bits"])


@pytest.mark.gpu
def test_gpu_match_matches_reference_vectors(gpu_ctx, pin):
    m = gpu_ctx.match(pin["match_q"], pin["match_t"])
    assert np.array_equal(m["left_idx"], pin["match_left"])
    assert np.array_equal(m["right_idx"], pin["match_right"])
    pairs, _ = gpu_ctx.match_mutual(pin["match_q"], pin["match_t"])
    assert np.array_equal(pairs, pin["match_pairs"])


@pytest.mark.gpu
def test_gpu_descriptor_flow_matches_reference_vectors(bshot, synth, pin):
    """two frames through one context like the reference's persistent `cb`: REFERENCE normals placement incl. the
    stale [K1, K0) entries; north_star tolerance: >= 99.9 % identical B-SHOT bits, LRF within 1e-4"""
    f0, f1 = flow_frames(synth, pin)
    with bshot.Context(0, max_points=16384, max_keypoints=128, max_targets=128) as ctx:
        ctx.set_cloud(f0)
        ctx.set_keypoints(pin["flow_kp0"])
        n0 = ctx.compute_normals(bshot.NORMALS_REFERENCE, 3000.0, 300)
        d0 = ctx.compute_shot(3000.0)
        ctx.set_cloud(f1)
        ctx.set_keypoints(pin["flow_kp1"])
        n1 = ctx.compute_normals(bshot.NORMALS_REFERENCE, 3000.0, 300)
        d1 = ctx.compute_shot(3000.0)
    same0 = (synth.unpack_bits(d0["bits"]) == synth.unpack_bits(pin["flow_bits0"])).mean()
    same1 = (synth.unpack_bits(d1["bits"]) == synth.unpack_bits(pin["flow_bits1"])).mean()
    assert same0 >= 0.999 and same1 >= 0.999, (same0, same1)
    fin = np.isfinite(pin["flow_rf0"]).all(1)
    assert np.array_equal(np.isfinite(d0["rf"]).all(1), fin)
    assert np.abs(d0["rf"][fin] - pin["flow_rf0"][fin]).max() <= 1e-4
    # placement: rows [0,96) of frame 0 hold keypoint normals, the rest zeros; frame 1 keeps rows [64,96) of frame 0
    assert np.allclose(n0[:96, :3], pin["flow_normals0_head"][:96, :3], atol=2e-3, equal_nan=True)
    assert not n0[96:128].any()
    assert np.array_equal(n1[64:96], n0[64:96], equal_nan=True)
    assert np.allclose(n1[:64, :3], pin["flow_normals1_head"][:64, :3], atol=2e-3, equal_nan=True)
