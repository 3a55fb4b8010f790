"""CPU checks of the float64 SHOT reference (tests/shot_f64.py) and of its GPU-vs-reference checker:
agreement with the fp32 oracle and the numpy restatement on small clouds, the exact half-radius shell test, and
checker mutations that must fail."""
import numpy as np
import pytest

import shot_f64 as sf
from shot_numpy import lrf_numpy, shot_numpy

f32 = np.float32
SHELL_RADII = [3000.1, 2999.7, 1234.567, 2500.3]


def blob(n, seed, scale=(1200.0, 700.0, 300.0)):
    rng = np.random.default_rng(seed)
    pts = (rng.normal(0, 1, (n, 3)) * scale).astype(f32)
    nrm = rng.normal(0, 1, (n, 4)).astype(f32)
    nrm[:, :3] /= np.linalg.norm(nrm[:, :3], axis=1, keepdims=True).astype(f32)
    return pts, nrm


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("R", [700.0, 1500.0, 3000.0, 1234.567])
def test_reference_matches_oracle_and_numpy(oracle, seed, R):
    pts, nrm = blob(500, seed, (R / 2, R / 3, R / 6))
    nrm[::7, 1] = np.nan                                         # invalid normals are skipped
    oc = oracle.Cloud(pts)
    for q in pts[:6]:
        L = sf.lrf_f64(pts, q, R)
        rf_o, nv_o = oc.lrf(q[None], R)
        rf_n, nv_n = lrf_numpy(pts, q, R)
        assert L["n_valid"] == nv_o[0] == nv_n
        assert np.abs(L["rf"] - rf_o[0]).max() <= 1e-6 and np.abs(L["rf"] - rf_n).max() <= 1e-6
        ref = sf.shot_f64(pts, q, R, nrm, L["rf"])
        so, _, nn, _ = oc.shot(q[None], nrm, R, rf_in=L["rf"][None])
        assert ref["n_all"] == nn[0]
        # a few hundred fp32 votes per descriptor: the oracle's running sums agree to ~1e-7
        assert np.abs(so[0] - ref["hist"]).max() <= 1e-6
        assert np.abs(shot_numpy(pts, q, R, nrm, L["rf"]) - ref["hist"]).max() <= 1e-6
        assert np.array_equal(ref["support"], ref["raw"] != 0)
        c = sf.check_shot(so[0], oracle.bshot(so), ref, sf.fx_bits(ref["n_all"]))
        assert c["ok"], c["why"]


def test_nibbles_match_the_oracle_binariser(oracle):
    rng = np.random.default_rng(4)
    shot = rng.random((300, 352)).astype(f32)
    shot[rng.random(shot.shape) < 0.6] = 0.0
    shot[7] = np.nan
    assert np.array_equal(sf.nibbles(shot), sf.bits_nibbles(oracle.bshot(shot)))


def shell_cloud(R, x):
    """keypoint at the origin, a neighbour at (x, 0, 0) and four others well inside / outside the shell"""
    pts = np.array([[0, 0, 0], [x, 0, 0], [0.2 * R, 0.1 * R, 0.05 * R], [-0.3 * R, 0.2 * R, -0.1 * R],
                    [0.1 * R, -0.7 * R, 0.2 * R], [-0.2 * R, -0.1 * R, 0.8 * R]], f32)
    nrm = np.zeros((len(pts), 4), f32)
    nrm[:, 2] = 1.0
    return pts, nrm


@pytest.mark.parametrize("R", SHELL_RADII)
def test_shell_boundary_is_outer(oracle, R):
    """a neighbour at sqd == fl(R^2/4) where fp32 rounds R^2/4 UP lies beyond R/2: PCL puts it in the outer shell"""
    quarter = float(f32(R)) ** 2 / 4.0
    up = float(f32(quarter))
    assert up > quarter                                         # these radii round R^2/4 up
    x = f32(R / 2)
    assert float(x * x) == up                                   # ... and the planted neighbour sits on that value
    pts, nrm = shell_cloud(R, x)
    rf = np.array([1, 0, 0, 0, 1, 0, 0, 0, 1], f32)
    with_p = sf.shot_f64(pts, pts[0], R, nrm, rf)
    without = sf.shot_f64(np.delete(pts, 1, 0), pts[0], R, np.delete(nrm, 1, 0), rf)
    votes = with_p["raw"] - without["raw"]
    # (x, 0, 0) with an axis-aligned rf: sector volume 12 (inner) / 14 (outer), normal along z -> shape bin 10;
    # the neighbour's own-bin weight (> 2) goes to the outer volume, the radial half-vote (0.5) to the inner one
    assert votes[14 * 11 + 10] > 2.0 and abs(votes[12 * 11 + 10] - 0.5) < 1e-6
    so, _, _, _ = oracle.Cloud(pts).shot(pts[:1], nrm, R, rf_in=rf[None])
    assert np.abs(so[0] - with_p["hist"]).max() <= 1e-6


def checker_case(n=2000, seed=5):
    pts, nrm = blob(n, seed)
    q = pts[0]
    L = sf.lrf_f64(pts, q, 3000.0)
    ref = sf.shot_f64(pts, q, 3000.0, nrm, L["rf"])
    return ref, sf.fx_bits(ref["n_all"])


def test_checker_accepts_the_reference_in_fp32():
    ref, fx = checker_case()
    g = ref["hist"].astype(f32)
    c = sf.check_shot(g, None, ref, fx)
    assert c["ok"] and c["excess"] < 0.1, c


def test_checker_rejects_a_moved_vote():
    """one vote of weight 1e-3 moved from the fullest bin to another populated bin"""
    ref, fx = checker_case()
    raw = ref["raw"].copy()
    a = int(np.argmax(raw))
    b = int(np.nonzero(ref["support"])[0][np.argsort(raw[ref["support"]])[len(raw[ref["support"]]) // 2]])
    assert a != b
    raw[a] -= 1e-3
    raw[b] += 1e-3
    g = (raw / np.sqrt(np.sum(raw * raw))).astype(f32)
    c = sf.check_shot(g, None, ref, fx)
    assert not c["ok"] and ("bin %d" % a in c["why"] or "bin %d" % b in c["why"]), c


def test_checker_rejects_support_and_bits_errors():
    ref, fx = checker_case()
    empty = int(np.nonzero(ref["votes"] == 0)[0][0])
    g = ref["hist"].astype(f32)
    g[empty] = 1e-30                                              # a vote where no neighbour can vote
    assert not sf.check_shot(g, None, ref, fx)["ok"]
    g = ref["hist"].astype(f32)
    bits = np.zeros((1, 6), np.uint64)
    j = int(np.argmax(np.abs(ref["hist"]).reshape(88, 4).sum(1)))  # a nibble far from the thresholds? flip to 0xF
    want = sf.nibbles(g)
    bits[0, (4 * j) // 64] = np.uint64((want[j] ^ 0xF) << ((4 * j) % 64))
    for i in range(88):
        if i != j:
            bits[0, (4 * i) // 64] |= np.uint64(int(want[i]) << ((4 * i) % 64))
    c = sf.check_shot(g, bits, ref, fx)
    near = sf.near_threshold(ref["hist"], sf.bound(ref, fx))[j]
    assert c["ok"] == bool(near) and (near or "nibble %d" % j in c["why"]), c


def test_fp32_oracle_at_1e5_neighbours(oracle):
    """The fp32 oracle sums ~1e5 votes in neighbour order.  Measured against the float64 reference its error is far
    above the reference's own fp32 rounding, so it is the worse judge of the kernel; it still stays inside the
    kernel's fixed-point bound at fx_bits = 13 (that bound is a worst case, the oracle's rounding a random walk)."""
    pts, nrm = blob(100000, 6)
    q = pts[0]
    L = sf.lrf_f64(pts, q, 3000.0)
    ref = sf.shot_f64(pts, q, 3000.0, nrm, L["rf"])
    fx = sf.fx_bits(ref["n_all"])
    assert ref["n_all"] > 80000 and fx == 13
    so, _, _, _ = oracle.Cloud(pts).shot(q[None], nrm, 3000.0, rf_in=L["rf"][None])
    oracle_err = np.abs(so[0] - ref["hist"]).max()
    cast_err = np.abs(ref["hist"].astype(f32) - ref["hist"]).max()
    assert oracle_err > 5 * cast_err, (oracle_err, cast_err)
    c = sf.check_shot(so[0], None, ref, fx)
    assert c["ok"], c["why"]


def test_reference_speed_at_2e6_neighbours():
    import time
    pts, nrm = blob(2_000_000, 7)
    t = time.perf_counter()
    q = np.zeros(3, f32)
    L = sf.lrf_f64(pts, q, 3000.0)
    ref = sf.shot_f64(pts, q, 3000.0, nrm, L["rf"])
    assert ref["n_all"] > 1_900_000 and sf.fx_bits(ref["n_all"]) == 9
    assert time.perf_counter() - t < 30.0


def tie_set(m, shell, seed, pref, R=3000.0):
    """points closed under (x, y, z) -> (+-x, +-y, +-z), no zero coordinate, axis spreads ~ 1 : 0.5 : 0.2.
    shell: all radii within +-0.1 % of 0.502 R (one tie-histogram bin of width R^2/256 holds them all).
    The sign variants inside each equal-sqd group of 8 are ordered so that the five keys around the median rank
    take the variants `pref` in turn.  Index 0 is the keypoint (the origin)."""
    rng = np.random.default_rng(seed)
    base = rng.uniform(0.5, 1.0, (m, 3)) * [1.0, 0.5, 0.2]
    if shell:
        base *= (0.502 * R * rng.uniform(0.999, 1.001, (m, 1))) / np.linalg.norm(base, axis=1, keepdims=True)
    else:
        base *= R * rng.uniform(0.15, 0.9, (m, 1)) / np.linalg.norm(base, axis=1, keepdims=True)
    base = base.astype(f32)
    sq = (base.astype(np.float64) ** 2).sum(1)
    base = base[np.argsort(sq)]
    signs = np.array([(sx, sy, sz) for sx in (1, -1) for sy in (1, -1) for sz in (1, -1)], f32)
    n = 8 * m
    med = n // 2
    window = {r: pref[r - (med - 2)] for r in range(med - 2, med + 3)}
    pts = [np.zeros(3, f32)]
    for g in range(m):
        order = [None] * 8
        for r, v in window.items():
            if r // 8 == g:
                order[r % 8] = v
        rest = [s for s in map(tuple, signs) if s not in order]
        order = [o if o is not None else rest.pop(0) for o in order]
        pts += [base[g] * np.asarray(o, f32) for o in order]
    return np.asarray(pts, f32)


# five median keys: x majority negative (3 of 5), z majority positive (4 of 5); and the mirror case
PREF_A = [(-1, 1, 1), (-1, -1, 1), (1, 1, 1), (-1, 1, -1), (1, -1, 1)]
PREF_B = [(1, 1, -1), (1, -1, -1), (-1, 1, -1), (1, 1, 1), (-1, -1, -1)]


@pytest.mark.parametrize("shell", [False, True])
@pytest.mark.parametrize("pref", [PREF_A, PREF_B])
def test_tie_sets_tie_and_follow_the_median_five(oracle, shell, pref):
    pts = tie_set(80 if shell else 6, shell, 3, pref)
    L = sf.lrf_f64(pts, pts[0], 3000.0)
    assert L["tie"] == (True, True) and L["s"] == (0, 0)
    assert min(L["gaps"]) > 0.1
    sx = -1 if sum(p[0] < 0 for p in pref) >= 3 else 1
    sz = -1 if sum(p[2] < 0 for p in pref) >= 3 else 1
    assert np.allclose(L["rf"][[0, 8]], [sx, sz], atol=1e-6)
    rf_o, _ = oracle.Cloud(pts).lrf(pts[:1], 3000.0)
    assert np.abs(rf_o[0] - L["rf"]).max() <= 1e-6
    if shell:
        sqd = (pts[1:].astype(np.float64) ** 2).sum(1)
        bins = np.minimum(255, (sqd * 256 / 3000.0 ** 2).astype(int))
        assert len(set(bins)) == 1 and len(bins) > 512
