"""Float64 reference of SHOT352 and the SHOT LRF for one keypoint, vectorised numpy.

The CUDA kernel (csrc/shot.cu) and the CPU oracle both sum fp32 votes; at 10^5 neighbours the oracle's fp32
running sums in neighbour order carry ~1e-3 relative error of their own and cannot judge the kernel.  This
reference takes every DECISION on exactly the values PCL compares (fp32 squared distance against fl(R^2), fp32
dot products with the |.| < 1e-30 clamp, the double shape bin, the sector bits, the exact `sqd > R^2/4` shell
test) and computes the weights and the sums in float64.

`check_shot` compares a kernel descriptor with the reference through a per-bin bound derived from the bin's vote
count (see its docstring); `nibbles` restates B-SHOT's binariser (include/bshot_bits.h:160-260)."""
import numpy as np

f32, f64 = np.float32, np.float64
RAD_45, RAD_90, RAD_135, RAD_PI_7_8 = np.pi / 4, np.pi / 2, 3 * np.pi / 4, 7 * np.pi / 8
EPS32 = 2.0 ** -24

# Per-vote error of the kernel's fp32 interpolation weights (csrc/shot.cu, default build), before the elevation
# term that `shot_f64` adds per neighbour:
#   shape   fbin = (float)(bin - step) from the same double bin: <= 2^-25 |fbin|                  ~ 3e-8
#   radial  rd = (fl(sqrt sqd) - fl(3R/4 or R/4)) * fl(2/R): three roundings of values <= R,
#           scaled by 2/R, plus the product's rounding: <= ~6 * 2^-24                              ~ 4e-7
#   elev.   acos_poly: A&S 4.4.46 (2e-8) evaluated in fp32 near pi/2, < 2.5e-7 rad; times 2/pi     ~ 2e-7
#   azim.   atan_sector < 4e-8 rad; the fp32 sector rotation (cos/sin 22.5 deg to 2^-24) and the
#           ratio yq/xq (|t| <= 0.41) add ~1e-7 rad; the atan2f fall-back ~6e-7 rad; times 4/pi   <= 8e-7
#   own     w = 1 - |fbin| + 1 - |rd| + 1 - |id| + 1 - |ad|: the four errors above plus 7 fp32
#           roundings of values <= 4 (7 * 2^-22 ~ 1.7e-6 worst case, ~4e-7 typical)
# 1e-6 covers every vote but the worst-case own-bin sum; WEIGHT_ERR_OWN covers that one.
WEIGHT_ERR = 1e-6
WEIGHT_ERR_OWN = 3e-6
# inc_cos = zr / dist in fp32 (fl(sqrt) and the division): relative error <= 2 * 2^-24 + rounding of the clamp
INC_COS_REL = 3 * EPS32


def fdot3(a, b):
    """(a0*b0 + a1*b1) + a2*b2 in fp32 without contraction, rows of a against vector b"""
    a = np.asarray(a, f32)
    b = np.asarray(b, f32)
    return ((a[..., 0] * b[0]) + (a[..., 1] * b[1])) + (a[..., 2] * b[2])


def neighbourhood(pts, q, R):
    """fp32 differences and squared distances (FLANN L2_Simple, no FMA), the `sqd < fl(R^2)` mask"""
    pts = np.asarray(pts, f32)
    q = np.asarray(q, f32)
    d = (pts - q).astype(f32)
    sqd = ((d[:, 0] * d[:, 0]) + (d[:, 1] * d[:, 1])) + (d[:, 2] * d[:, 2])
    R2 = f32(float(f32(R)) * float(f32(R)))
    with np.errstate(invalid="ignore"):
        inside = sqd < R2
    if not np.isfinite(q).all():
        inside[:] = False
    return d, sqd, inside


def lrf_f64(pts, q, R):
    """SHOTLocalReferenceFrameEstimation::getLocalRF in float64 (numpy.linalg.eigh).
    Returns dict(rf (9,) fp32 as PCL stores it, n_valid, s (pre-tie votes of x and z), tie (bool per axis),
    gaps (relative eigen-gaps (l2 - l1)/l2, (l1 - l0)/l2), median5 (indices at ranks median-2..median+2))."""
    d, sqd, inside = neighbourhood(pts, q, R)
    q = np.asarray(q, f32)
    idx = np.nonzero(inside & ~(np.asarray(pts, f32) == q).all(1))[0]
    idx = idx[np.lexsort((idx, sqd[idx]))]                       # ordered by (sqd, index)
    nv = len(idx)
    out = dict(rf=np.full(9, np.nan, f32), n_valid=nv, s=(0, 0), tie=(False, False), gaps=(np.nan, np.nan), median5=None)
    if nv < 5:
        return out
    v = d[idx].astype(f64)
    w = float(f32(R)) - np.sqrt(sqd[idx].astype(f64))
    cov = (v * w[:, None]).T @ v / w.sum()
    ev, V = np.linalg.eigh(cov)
    if not np.isfinite(ev).all():
        return out
    x, z = V[:, 2].copy(), V[:, 0].copy()
    med = nv // 2
    five = idx[med - 2: med + 3]
    vf = v[med - 2: med + 3]
    s_all, ties = [], []
    for ax in (x, z):
        s = 2 * int((v @ ax >= 0).sum()) - nv
        s_all.append(s)
        ties.append(s == 0)
        if s == 0:
            if int((vf @ ax > 0).sum()) < 3:
                ax *= -1
        elif s < 0:
            ax *= -1
    xf, zf = x.astype(f32), z.astype(f32)
    yf = np.array([zf[1] * xf[2] - zf[2] * xf[1], zf[2] * xf[0] - zf[0] * xf[2], zf[0] * xf[1] - zf[1] * xf[0]], f32)
    out.update(rf=np.concatenate([xf, yf, zf]).astype(f32), s=tuple(s_all), tie=tuple(ties),
               gaps=((ev[2] - ev[1]) / ev[2], (ev[1] - ev[0]) / ev[2]), median5=five)
    return out


def _acos_spread(c, dc):
    """largest |acos(c') - acos(c)| over |c' - c| <= dc, c' clamped to [-1, 1] (acos is monotone)"""
    a = np.arccos(c)
    return np.maximum(np.abs(np.arccos(np.clip(c - dc, -1.0, 1.0)) - a), np.abs(np.arccos(np.clip(c + dc, -1.0, 1.0)) - a))


def shot_f64(pts, q, R, normals4, rf):
    """SHOTEstimation::computePointSHOT for one keypoint with the given rf, weights and sums in float64.

    Returns dict with
      hist     (352,) float64 normalised histogram (NaN when PCL gives a NaN descriptor)
      raw      (352,) float64 histogram before normalisation
      votes    (352,) int, votes a bin can receive: PCL's votes (zero weights included) plus, where the kernel's
               fp32 weight decides a direction that PCL decides in double and the weight is within its error of
               zero, the vote the other direction would give
      err      (352,) float64, sum of the per-vote weight errors of those votes (the fixed-point term is added by
               `bound`, which knows fx_bits)
      support  (352,) bool, bins with a non-zero vote
      n_all, n_valid"""
    pts = np.asarray(pts, f32)
    q = np.asarray(q, f32)
    rf = np.asarray(rf, f32).reshape(9)
    d, sqd, inside = neighbourhood(pts, q, R)
    n_all = int(inside.sum())
    n_valid = int((inside & ~(pts == q).all(1)).sum())
    res = dict(hist=np.full(352, np.nan), raw=np.zeros(352), votes=np.zeros(352, np.int64), err=np.zeros(352),
               support=np.zeros(352, bool), n_all=n_all, n_valid=n_valid)
    if n_all < 5 or not np.isfinite(rf).all() or not np.isfinite(q).all():
        return res
    idx = np.nonzero(inside)[0]
    nrm = np.asarray(normals4, f32)[idx, :3]
    keep = np.isfinite(nrm).all(1)
    idx, nrm = idx[keep], nrm[keep]
    sq = sqd[idx].astype(f64)
    dist = np.sqrt(sq)
    keep = ~(np.abs(dist) < 1e-15)
    idx, nrm, sq, dist = idx[keep], nrm[keep], sq[keep], dist[keep]
    dd = d[idx]
    Rf = float(f32(R))

    cosine = np.clip(fdot3(nrm, rf[6:9]).astype(f64), -1.0, 1.0)
    bin_ = ((1.0 + cosine) * 10) / 2
    xr = fdot3(dd, rf[0:3]).astype(f64)
    yr = fdot3(dd, rf[3:6]).astype(f64)
    zr = fdot3(dd, rf[6:9]).astype(f64)
    xr[np.abs(xr) < 1e-30] = 0.0
    yr[np.abs(yr) < 1e-30] = 0.0
    zr[np.abs(zr) < 1e-30] = 0.0
    bit4 = ((yr > 0) | ((yr == 0) & (xr < 0))).astype(np.int64)
    bit3 = np.where((xr > 0) | ((xr == 0) & (yr > 0)), 1 - bit4, bit4)
    desc = ((bit4 << 3) + (bit3 << 2)) << 1
    first = (xr * yr > 0) | (xr == 0)
    desc += np.where(first, np.where(np.abs(xr) >= np.abs(yr), 0, 4), np.where(np.abs(xr) > np.abs(yr), 4, 0))
    desc += (zr > 0).astype(np.int64)
    outer = sq > (Rf * Rf) / 4.0                          # exact: R*R is exact in double, /4 too
    desc += np.where(outer, 2, 0)
    step = np.floor(bin_ + 0.5).astype(np.int64)
    vol = desc * 11
    beta = bin_ - step

    tgt, wt, er = [], [], []                              # vote targets, float64 weights, per-vote weight errors

    def vote(t, w, e):
        tgt.append(np.asarray(t, np.int64))
        wt.append(np.asarray(w, f64))
        er.append(np.broadcast_to(np.asarray(e, f64), np.shape(t)))

    def vote_dir(mask_pos, t_pos, t_neg, w, close, e):
        """direction decided by a sign the kernel evaluates in fp32 (PCL: in double): PCL's vote, plus a
        zero-weight vote at the other target where the deciding value `close` is within its error of zero"""
        vote(np.where(mask_pos, t_pos, t_neg), w, e)
        near = close <= e
        if near.any():
            vote(np.where(mask_pos, t_neg, t_pos)[near], np.zeros(int(near.sum())), e[near])

    w_own = 1.0 - np.abs(beta)
    # shape: the double bin is the kernel's too, no phantom needed; beta == 0 gives PCL's zero vote to step - 1
    vote(np.where(beta > 0, vol + (step + 1) % 10, vol + (step + 9) % 10), np.abs(beta), WEIGHT_ERR)
    # radial
    rd = np.where(outer, (dist - 0.75 * Rf) / (Rf / 2), (dist - 0.25 * Rf) / (Rf / 2))
    w_own += 1.0 - np.abs(rd)
    to_nb = np.where(outer, ~(dist > 0.75 * Rf), ~(dist < 0.25 * Rf))
    nb_rad = np.where(outer, desc - 2, desc + 2) * 11 + step
    vote_dir(to_nb, nb_rad, -1, np.where(to_nb, np.abs(rd), 0.0), np.abs(rd), np.full(len(idx), WEIGHT_ERR))
    # elevation: PCL's `inc > 90 deg || (|inc - 90 deg| < 1e-30 && z <= 0)` is z <= 0 for a monotone acos
    inc_cos = np.clip(zr / dist, -1.0, 1.0)
    inc = np.arccos(inc_cos)
    lower = ~(zr > 0)
    idv = np.where(lower, (inc - RAD_135) / RAD_90, (inc - RAD_45) / RAD_90)
    w_own += 1.0 - np.abs(idv)
    e_inc = WEIGHT_ERR + _acos_spread(inc_cos, INC_COS_REL * np.abs(inc_cos) + EPS32) / RAD_90
    to_nb = np.where(lower, ~(inc > RAD_135), ~(inc < RAD_45))
    nb_el = np.where(lower, desc + 1, desc - 1) * 11 + step
    vote_dir(to_nb, nb_el, -1, np.where(to_nb, np.abs(idv), 0.0), np.abs(idv), e_inc)
    # azimuth
    has_az = (yr != 0) | (xr != 0)
    az = np.arctan2(yr, xr)
    sel = desc >> 2
    ad = np.clip((az - (-RAD_PI_7_8 + RAD_45 * sel)) / RAD_45, -0.5, 0.5)
    ad = np.where(has_az, ad, 0.0)
    w_own += np.where(has_az, 1.0 - np.abs(ad), 0.0)
    nb_az = np.where(ad > 0, (desc + 4) % 32, (desc + 28) % 32) * 11 + step
    alt_az = np.where(ad > 0, (desc + 28) % 32, (desc + 4) % 32) * 11 + step
    h = np.nonzero(has_az)[0]
    vote_dir(np.ones(len(h), bool), nb_az[h], alt_az[h], np.abs(ad[h]), np.abs(ad[h]), np.full(len(h), WEIGHT_ERR))
    # own bin
    vote(vol + step, w_own, WEIGHT_ERR_OWN + (e_inc - WEIGHT_ERR))

    t = np.concatenate(tgt)
    w = np.concatenate(wt)
    e = np.concatenate(er)
    real = t >= 0                                         # -1: "no neighbour vote" placeholder of vote_dir
    t, w, e = t[real], w[real], e[real]
    raw = np.bincount(t, weights=w, minlength=352)
    res["raw"] = raw
    res["votes"] = np.bincount(t, minlength=352)
    res["err"] = np.bincount(t, weights=e, minlength=352)
    res["support"] = np.bincount(t[w != 0], minlength=352) > 0
    norm = np.sqrt(np.sum(raw * raw))
    res["hist"] = raw / norm
    return res


def fx_bits(n_all):
    """the kernel's fixed-point resolution: largest b <= 28 with 2^b * 4.1 * n_all < 2^32"""
    return min(28, max(0, int(np.floor(np.log2(4294967295.0 / (4.1 * max(n_all, 1)))))))


def bound(ref, fxb):
    """per-bin bound on |g_b - r_b| for a kernel descriptor g against the reference r.
    Unnormalised: each vote to bin b is off by at most half a fixed-point quantum 2^-(fxb+1) plus its weight
    error, so |h_b - H_b| <= E_b = m_b 2^-(fxb+1) + err_b.  Normalised, with N = ||H|| and ||h - H|| <= ||E||:
    |h_b/||h|| - H_b/N| <= (E_b + |r_b| ||E||) / (N - ||E||), plus the fp32 conversion of the integer sum, the
    fp32 norm and the fp32 division (a few ulp of g_b)."""
    E = ref["votes"] * 2.0 ** -(fxb + 1) + ref["err"]
    N = float(np.sqrt(np.sum(ref["raw"] ** 2)))
    En = float(np.sqrt(np.sum(E * E)))
    r = np.abs(ref["hist"])
    assert En < 0.5 * N, "fixed-point and weight errors swamp the histogram"
    return (E + r * En) / (N - En) + 8 * EPS32 * r + 2.0 ** -140


def nibbles(shot):
    """B-SHOT's 4-float -> nibble rule on fp32 values (include/bshot_bits.h:160-260), (..., 352) -> (..., 88)"""
    v = np.asarray(shot, f32).reshape(*np.shape(shot)[:-1], 88, 4)
    a, b, c, d = (v[..., k] for k in range(4))
    t = 0.9 * (((a + b) + c) + d).astype(f64)
    conds = [a, b, c, d, a + b, b + c, c + d, a + d, b + d, a + c, (a + b) + c, (b + c) + d, (a + c) + d, (a + b) + d]
    codes = [0x1, 0x2, 0x4, 0x8, 0x3, 0x6, 0xC, 0x9, 0xA, 0x5, 0x7, 0xE, 0xD, 0xB]
    out = np.full(a.shape, 0xF, np.int64)
    done = (a == 0) & (b == 0) & (c == 0) & (d == 0)
    out[done] = 0
    for s, code in zip(conds, codes):
        hit = ~done & (s.astype(f64) > t)
        out[hit] = code
        done |= hit
    return out


def bits_nibbles(bits):
    """(K, 6) uint64 B-SHOT records -> (K, 88) nibbles"""
    b = np.asarray(bits, np.uint64).reshape(-1, 6)
    j = np.arange(88)
    return ((b[:, (4 * j) // 64] >> ((4 * j) % 64).astype(np.uint64)) & np.uint64(0xF)).astype(np.int64)


# the 14 subsets of a nibble that the binariser compares against 0.9 * sum, in its order
_SUBSETS = [(0,), (1,), (2,), (3,), (0, 1), (1, 2), (2, 3), (0, 3), (1, 3), (0, 2), (0, 1, 2), (1, 2, 3), (0, 2, 3), (0, 1, 3)]


def near_threshold(r, b):
    """(88,) bool: some threshold comparison of the nibble is within the bound (r: reference values, b: bounds)"""
    r = np.asarray(r, f64).reshape(88, 4)
    b = np.asarray(b, f64).reshape(88, 4)
    S, BS = r.sum(1), b.sum(1)
    near = np.zeros(88, bool)
    for sub in _SUBSETS:
        s = r[:, sub].sum(1)
        bs = b[:, sub].sum(1)
        near |= np.abs(s - 0.9 * S) <= bs + 0.9 * BS + 16 * EPS32 * S
    near |= (r == 0).all(1) | (r <= b).all(1)            # the all-zero test
    return near


def check_shot(g_shot, g_bits, ref, fxb):
    """Judge one kernel descriptor against the float64 reference.  Returns dict(ok, why, excess (max |g-r| / bound),
    maxdiff, nib_diff); `ok` is False with a reason on the first violated condition:
      values   |g_b - r_b| <= bound_b for every bin
      support  the kernel's non-zero bins are bins that can receive a vote; a reference bin with mass above its
               bound is non-zero in the kernel's descriptor
      bits     every nibble whose bits differ from the binarised reference has a threshold within the bound"""
    g = np.asarray(g_shot, f64)
    r = ref["hist"]
    out = dict(ok=True, why="", excess=0.0, maxdiff=0.0, nib_diff=0)
    if np.isnan(r).all():
        if not np.isnan(g).all():
            out.update(ok=False, why="reference NaN, kernel finite")
        return out
    if np.isnan(g).any():
        out.update(ok=False, why="kernel NaN, reference finite")
        return out
    bd = bound(ref, fxb)
    diff = np.abs(g - r)
    out["maxdiff"] = float(diff.max())
    out["excess"] = float((diff / bd).max())
    if (diff > bd).any():
        b = int(np.argmax(diff / bd))
        out.update(ok=False, why=f"bin {b}: |g-r| = {diff[b]:.3g} > bound {bd[b]:.3g} (g={g[b]:.9g} r={r[b]:.9g} votes={ref['votes'][b]})")
        return out
    if ((g != 0) & (ref["votes"] == 0)).any():
        out.update(ok=False, why="kernel support outside the reference's vote targets")
        return out
    if ((g == 0) & ref["support"] & (r > bd)).any():
        out.update(ok=False, why="reference bin above its bound missing from the kernel's support")
        return out
    if g_bits is not None:
        nr = nibbles(r.astype(f32))
        ng = bits_nibbles(g_bits)[0]
        dif = nr != ng
        out["nib_diff"] = int(dif.sum())
        if (dif & ~near_threshold(r, bd)).any():
            j = int(np.nonzero(dif & ~near_threshold(r, bd))[0][0])
            out.update(ok=False, why=f"nibble {j}: bits {ng[j]:x} vs reference {nr[j]:x} away from every threshold")
    return out
