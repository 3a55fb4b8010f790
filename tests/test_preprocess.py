"""Scan preprocessor (SURVEY 8f #4): bshot_preprocess against myslam::Preprocessor::run of the reference
(src/preprocess.cpp:213-223).  The checker is the reference's OWN source compiled unchanged (oracle/_ref/libbshot_ref.so,
built by oracle/Makefile `ref` where the reference sources are at hand).  Golden vectors made by it
(tests/golden/preprocess_pin.npz, tests/golden/make_preprocess_pin.py) hold on any machine.  The other device cases below
compare live with that library where it is built, and everywhere with a regression snapshot of the device output
(tests/golden/snapshots.py).  Bar: same number of points, the same coordinates bit for bit, in the same order."""
import os
import sys
import zlib

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
from make_preprocess_pin import CASES, lasers_crc  # noqa: E402
from snapshots import ExpectedPreprocessing, Snapshots  # noqa: E402


@pytest.fixture(scope="module")
def pin():
    return np.load(os.path.join(HERE, "golden", "preprocess_pin.npz"))


@pytest.fixture(scope="module")
def ref(oracle):
    if oracle.ref_lib() is None:
        pytest.skip("oracle/_ref/libbshot_ref.so not built (needs the reference sources at build time)")
    return oracle


@pytest.fixture(scope="module")
def expected(oracle, gpu_ctx):
    """what the device tests below must return (tests/golden/snapshots.py)"""
    snapshots = Snapshots()
    yield ExpectedPreprocessing(snapshots, oracle, gpu_ctx)
    snapshots.save()


def same_points(a, b):
    if hasattr(b, "check"):        # an expectation of tests/golden/snapshots.py
        b.check(a, "points")
        return
    assert a.shape == b.shape, f"{a.shape[0]} points, expected {b.shape[0]}"
    diff = (a.view(np.uint32) != b.view(np.uint32)).any(axis=1)
    assert not diff.any(), f"{int(diff.sum())} of {len(a)} points differ, first at {int(np.argmax(diff))}: {a[np.argmax(diff)]} vs {b[np.argmax(diff)]}"


def column(az, verts, dists):
    return dict(azimuth=np.full(len(verts), az, np.float64), vertical=np.asarray(verts, np.float64), distance=np.asarray(dists, np.uint16))


def cat(cols):
    return {k: np.concatenate([c[k] for c in cols]) for k in ("azimuth", "vertical", "distance")}


RING = np.array([-20.0, -15.0, -10.0, -5.0, 0.0, 5.0])


def ground_dist(vert_deg, height=2450.0):
    return np.round(height / np.sin(np.deg2rad(-np.asarray(vert_deg))) / 2.0)


# ---- the reference-compiled library itself (CPU) ------------------------------------------------------------------------
def test_generator_and_reference_still_give_the_golden_vectors(ref, synth, pin):
    for name, kw in CASES.items():
        L = synth.make_lasers(**kw)
        assert lasers_crc(L) == int(pin[name + "_crc"]), "the synthetic rotation changed: regenerate tests/golden/preprocess_pin.npz"
        same_points(ref.ref_preprocess(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"]), pin[name + "_xyz"])


def test_reference_removes_flat_ground_and_keeps_a_wall(ref):
    """known answer: beams that hit the plane 2450 mm under the sensor go, the ones that hit a wall stay"""
    down = RING[:4]
    cols = []
    for k in range(8):
        d = np.concatenate([ground_dist(down), [0, 0]])
        if k >= 4:  # a wall 6 m ahead seen by the three upper beams
            d[3:] = np.round(6000.0 / np.cos(np.deg2rad(RING[3:])) / 2.0)
        cols.append(column(10.0 + 0.2 * k, RING, d))
    L = cat(cols)
    out = ref.ref_preprocess(L["azimuth"], L["vertical"], L["distance"], RING)
    # the first wall column keeps only its -5 degree beam: on the two rings that had no return before, the occlusion pass
    # compares against the first column of the scan (range 0 there, 0.8 degrees away) and drops the far side (:179-188)
    assert len(out) == 1 + 3 * 3
    horizontal = np.hypot(out[:, 0], out[:, 1])
    assert np.all(np.abs(horizontal - 6000.0) < 3.0)


def test_make_lasers_shape(synth):
    L = synth.make_lasers("hdl32e", 0, firings=50)
    assert L["azimuth"].shape == L["vertical"].shape == L["distance"].shape == (50 * 32,)
    assert L["distance"].dtype == np.uint16 and (np.diff(L["azimuth"]) < 0).sum() == 0
    W = synth.make_lasers("hdl32e", 0, firings=200, start_deg=350.0)
    assert (np.diff(W["azimuth"]) < 0).sum() == 1, "the sweep wraps through 0 degrees once (firing order, not sorted)"


# ---- the device path ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_gpu_matches_reference_made_vectors(gpu_ctx, synth, pin, name):
    L = synth.make_lasers(**CASES[name])
    assert lasers_crc(L) == int(pin[name + "_crc"])
    same_points(gpu_ctx.preprocess(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"]), pin[name + "_xyz"])


@pytest.mark.gpu
@pytest.mark.parametrize("sensor,frame", [("hdl32e", 0), ("hdl32e", 5), ("hdl64e", 1)])
def test_gpu_matches_reference_on_a_full_rotation(gpu_ctx, expected, synth, sensor, frame):
    L = synth.make_lasers(sensor, frame)
    want = expected.preprocess(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"])
    assert 0.2 * L["distance"].size < len(want) < 0.9 * L["distance"].size   # the ground is a large part of the scan
    same_points(gpu_ctx.preprocess(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"]), want)
    # the same rotation sorted the way `capture.retrieve(lasers, true)` sorts it: nothing changes
    o = np.lexsort((np.arange(L["azimuth"].size), L["azimuth"]))
    same_points(gpu_ctx.preprocess(L["azimuth"][o], L["vertical"][o], L["distance"][o], L["ring_deg"]), want)


@pytest.mark.gpu
def test_gpu_other_thresholds(gpu_ctx, expected, synth):
    L = synth.make_lasers("hdl32e", 3)
    for vert_init, lowpt in ((-0.6, -1700.0), (-0.55, -2200.0), (-0.7, -1950.0)):
        want = expected.preprocess(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], vert_init, lowpt)
        same_points(gpu_ctx.preprocess(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], vert_init, lowpt), want)


@pytest.mark.gpu
def test_gpu_edge_cases(gpu_ctx, expected, bshot):
    rng = np.random.default_rng(5)
    empty = gpu_ctx.preprocess(np.zeros(0), np.zeros(0), np.zeros(0, np.uint16), RING)
    assert empty.shape == (0, 3)

    def both(L, ring=RING):
        want = expected.preprocess(L["azimuth"], L["vertical"], L["distance"], ring)
        same_points(gpu_ctx.preprocess(L["azimuth"], L["vertical"], L["distance"], ring), want)
        return want

    # one column only; a column of lost returns; the known-answer wall
    both(column(33.0, RING, [3000, 3000, 3000, 3000, 3000, 3000]))
    both(cat([column(1.0, RING, [0] * 6), column(1.2, RING, [4000] * 6)]))
    # the same (azimuth, vertical) key twice: the later return replaces the earlier one (std::map assignment), also across
    # two separate runs of the same azimuth
    a = column(50.0, [-10.0, 0.0, -10.0, 5.0], [2500, 2600, 4100, 2700])
    b = column(50.2, RING, [4000] * 6)
    again = column(50.0, [0.0], [5200])
    w = both(cat([a, b, again]))
    assert len(w) > 0
    # descending azimuths, random order of the beams inside a firing, a beam below the start angle (vert_init = -0.6 rad =
    # -34.4 deg: then the FIRST map entry, which the ground pass skips, is that beam and the start entry is walked as a return)
    ring = np.array([-40.0, -20.0, -10.0, 0.0, 10.0])
    cols = []
    for k in range(40):
        p = rng.permutation(5)
        cols.append(column(300.0 - 0.3 * k, ring[p], rng.integers(0, 9000, 5)[p]))
    both(cat(cols), ring)
    # occlusion: a near pole in front of a far wall, both directions of the range jump, lost returns in between
    cols = []
    for k in range(60):
        d = np.full(6, 20000 // 2)
        if 20 <= k < 26:
            d[:] = 4000 // 2
        if k in (19, 26, 27):
            d[2:4] = 0
        cols.append(column(100.0 + 0.17 * k, RING, d))
    w = both(cat(cols))
    assert len(w) < 60 * 6
    # no ring table: the occlusion pass has nothing to walk
    L = cat(cols)
    same_points(gpu_ctx.preprocess(L["azimuth"], L["vertical"], L["distance"], np.zeros(0)), expected.preprocess(L["azimuth"], L["vertical"], L["distance"], np.zeros(0)))
    # random soup: arbitrary double azimuths incl. negative and -0.0 / +0.0 as one key
    n = 5000
    az = rng.choice(np.concatenate([rng.uniform(-5.0, 5.0, 300), [0.0, -0.0]]), n)
    L = dict(azimuth=az, vertical=rng.choice(RING, n), distance=rng.integers(0, 30000, n).astype(np.uint16))
    both(L)


@pytest.mark.gpu
def test_gpu_point_selection(gpu_ctx, expected, synth):
    """setSelectedPoints / haveSelectList / saveSelectPoints (test/odometry_test.cpp:144-160): selected returns only, or
    everything but them; an unsorted list with a duplicate (the cursor of readFrame stops advancing at it)"""
    L = synth.make_lasers("hdl32e", 1, firings=400, start_deg=200.0)
    n = L["azimuth"].size
    rng = np.random.default_rng(2)
    args = (L["azimuth"], L["vertical"], L["distance"], L["ring_deg"])
    everything = expected.preprocess(*args)
    for sel in (np.arange(0, n, 3), rng.permutation(n)[: n // 2], np.array([5, 900, 900, 4000, 7000]), np.zeros(0, np.int32), np.array([n + 5, -3, 10])):
        for save in (True, False):
            want = expected.preprocess(*args, select=sel, save_selected=save)
            same_points(gpu_ctx.preprocess(*args, select=sel, save_selected=save), want)
        kept = len(expected.preprocess(*args, select=sel, save_selected=True)) + len(expected.preprocess(*args, select=sel, save_selected=False))
        assert kept == len(everything)
    # no list but "save the unselected": nothing is written
    assert len(gpu_ctx.preprocess(*args, save_selected=False)) == len(expected.preprocess(*args, save_selected=False)) == 0


@pytest.mark.gpu
def test_gpu_capacity_errors(gpu_ctx, bshot):
    import ctypes as C
    L = cat([column(10.0 + 0.2 * k, RING, [3000] * 6) for k in range(10)])
    out = np.empty((4, 3), np.float32)
    n = C.c_size_t()
    rc = bshot.lib().bshot_preprocess(gpu_ctx.h, L["azimuth"].ctypes.data, L["vertical"].ctypes.data, L["distance"].ctypes.data, L["azimuth"].size,
                                      RING.ctypes.data, RING.size, -0.6, -1950.0, out.ctypes.data, 4, C.byref(n))
    assert rc == -2 and n.value > 4   # BSHOT_E_CAPACITY
    # more distinct vertical angles in one column than a column holds
    m = 200
    big = column(7.0, np.linspace(-30, 10, m), [3000] * m)
    with pytest.raises(bshot.BshotError):
        gpu_ctx.preprocess(big["azimuth"], big["vertical"], big["distance"], RING)
