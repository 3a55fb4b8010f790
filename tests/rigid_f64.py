"""Float64 reference of the rigid fits (ICP's and RANSAC's Procrustes step), numpy / scipy only.

The device kernels (csrc/icp.cu, csrc/ransac.cu) and the CPU oracle share one restatement of pcl::umeyama, so a
mistake in it passes every device == oracle test.  This module restates the fit from the definitions instead:

* `umeyama_f64` -- Umeyama without scaling in float64 with numpy's SVD and pcl::umeyama's rank rule
  (isMuchSmallerThan(s_i, s_0) at `precision`: 1e-5 for ICP's float estimator, 1e-12 for RANSAC's double one);
  rank 2 takes its sign from det U det V, every other rank from det Sigma.  It also returns the optimum of the
  Procrustes objective, max over proper rotations of tr(R^T Sigma), which is unique even where R is not.
* `icp_step_f64` / `icp_f64` -- the ICP loop: float64 nearest targets with the gap to the second-best target, the
  fit above, the mse; `icp_f64` restarts every step from the device's pose, bounds the fp32 drift of the device's
  points and flags a step whose nearest-target choice fp32 could flip.
* `ransac_f64` -- PCL's sampler replayed (mt19937 seeded 12345 through numpy, `>> 1`, the progressive shuffle),
  isSampleGood against a float64 sample_dist_thresh, float64 models and inlier counts, the adaptive stop and the
  in-order inliers.  Every decision fp32 could take the other way is flagged.
* `fit_bound` / `check_fit` -- judge a device transform against the reference with a bound built from the inputs
  (see `fit_bound`), and for rank <= 1 by what is unique: orthonormality, det +1, the objective and t = dm - R sm.
"""
import math

import numpy as np
from scipy.spatial import cKDTree

f32, f64 = np.float32, np.float64
U32, U64 = 2.0 ** -24, 2.0 ** -53
ICP_PRECISION, RANSAC_PRECISION = 1e-5, 1e-12


def gamma(k, u=U32):
    return k * u / (1.0 - k * u)


# ---- the Procrustes fit ---------------------------------------------------------------------------------------------
def umeyama_f64(src, dst, precision=ICP_PRECISION):
    """pcl::umeyama(src, dst, with_scaling = false) in float64 on the pairs (src[i], dst[i])."""
    s = np.asarray(src, f64).reshape(-1, 3)
    d = np.asarray(dst, f64).reshape(-1, 3)
    n = len(s)
    sm, dm = s.mean(0), d.mean(0)
    sigma = (d - dm).T @ (s - sm) / n
    if (d == d[0]).all() or (s == s[0]).all():   # one side is a single point: Sigma is exactly 0, whatever dm rounds to
        sigma = np.zeros((3, 3))
    U, sv, Vt = np.linalg.svd(sigma)
    det = float(np.linalg.det(sigma))
    rank = int(np.sum(~(sv <= sv[0] * precision))) if sv[0] > 0 else 0
    duv = float(np.sign(np.linalg.det(U) * np.linalg.det(Vt)))
    S = np.ones(3)
    if rank == 2:
        S[2] = duv
    elif rank == 3:
        S[2] = -1.0 if det < 0 else 1.0
    elif rank == 1:
        S[2] = duv          # one proper optimum; R is not unique here
    R = np.eye(3) if rank == 0 else U @ np.diag(S) @ Vt
    # max over SO(3) of tr(R^T Sigma): s0 + s1 + sign(det U det V) s2
    opt = float(sv[0] + sv[1] + duv * sv[2])
    return dict(R=R, t=dm - R @ sm, sv=sv, rank=rank, det=det, opt=opt, sigma=sigma, sm=sm, dm=dm, n=n,
                sign=duv if rank < 3 else S[2], s=s, d=d)


def fit_bound(fit, u=U32, k_sum=None, e_in=0.0, t_u=None):
    """Bound on |R_dev - R|_F and |t_dev - t| for a device fit of `fit`'s pairs.

    Sigma's entries are sums of products of rounded differences: with k_sum roundings on any summation path (ICP:
    ceil(n / 256) strided partial sums + the 8-level halving tree) and two more for the difference and the product,
    |dSigma_rc| <= (1/n) [sum_i (dd_ir |s_ic| + |d_ir| ds_ic) + gamma_{k+2} sum_i |d_ir| |s_ic|] + 2u |Sigma_rc|, where
    dd and ds are the errors of the centred coordinates: the centroid errors (gamma_{k+2} sum |x| / n, plus `e_in`, the
    error of the input source positions) and one rounding.  Then (special-orthogonal polar factor)
    |dR|_F <= 2 |dSigma|_F / (s1 + sign s2) plus the cast of R, and |dt| <= |ddm| + |dsm| + |dR|_F |sm| + rounding.
    At rank <= 1 R is not unique and dR bounds only |(R_dev - R) v0|, with s0 - s1 in the denominator."""
    s, d, n = fit["s"], fit["d"], fit["n"]
    if k_sum is None:
        k_sum = -(-n // 256) + 8
    g = gamma(k_sum + 2, u)
    dsm = g * np.abs(s).sum(0) / n + 2 * u * np.abs(fit["sm"]) + e_in
    ddm = g * np.abs(d).sum(0) / n + 2 * u * np.abs(fit["dm"])
    sc, dc = np.abs(s - fit["sm"]), np.abs(d - fit["dm"])
    ds = dsm + u * sc + e_in
    dd = ddm + u * dc
    dS = (dd.T @ (sc + ds) + dc.T @ ds + g * (dc + dd).T @ (sc + ds)) / n + 2 * u * np.abs(fit["sigma"])
    dS_f = float(np.linalg.norm(dS)) + 1e-13 * float(fit["sv"][0])
    sv = fit["sv"]
    den = sv[1] + fit["sign"] * sv[2]
    if fit["rank"] <= 1:   # R is not unique: dR bounds |(R_dev - R) v0| only, through the rotation of u0 and v0
        den = sv[0] - sv[1] if fit["rank"] == 1 else math.inf   # rank 0: R = I exactly
    dR = (2.0 * dS_f / den if den > 0 else math.inf) + math.sqrt(3.0) * U32 + 1e-12
    tu = U32 if t_u is None else t_u
    nsm, ndm = float(np.linalg.norm(fit["sm"])), float(np.linalg.norm(fit["dm"]))
    dt = (float(np.linalg.norm(ddm)) + float(np.linalg.norm(dsm)) + dR * nsm + gamma(4, tu) * (ndm + 2.0 * nsm)
          + 2 * U32 * float(np.linalg.norm(fit["t"])))
    dobj = 2.0 * math.sqrt(3.0) * dS_f + 2e-6 * float(sv[0])
    return dict(dSigma=dS_f, dR=dR, dt=dt, dobj=dobj, ddm=float(np.linalg.norm(ddm)), dsm=float(np.linalg.norm(dsm)))


def check_fit(R_dev, t_dev, fit, bound):
    """Judge a device rotation / translation against the float64 fit.  Full rank, or rank 2 at a proper optimum:
    |dR|_F and |dt| within `bound`.  Rank <= 1 (R not unique): R^T R = I within 1e-6, det R = +1, tr(R^T Sigma)
    within the bound of the optimum (plus the 2 (s1 + s2) the device may drop by calling the rank <= 1), and
    t = dm - R sm; at rank 0 also R = I, which the objective and t cannot tell from any other rotation.  Returns dict(ok, why, rR, rt) with the errors as fractions of their bounds."""
    R = np.asarray(R_dev, f64).reshape(3, 3)
    t = np.asarray(t_dev, f64).reshape(3)
    out = dict(ok=True, why="", rR=0.0, rt=0.0)

    def fail(msg):
        out["ok"] = False
        out["why"] = (out["why"] + "; " if out["why"] else "") + msg

    if not (np.isfinite(R).all() and np.isfinite(t).all()):
        fail(f"non-finite transform R={R.tolist()} t={t.tolist()}")
        return out
    orth = float(np.abs(R.T @ R - np.eye(3)).max())
    det = float(np.linalg.det(R))
    if orth > 1e-6:
        fail(f"R is not orthonormal: |R^T R - I| = {orth:.3g} (det {det:.3g}, R={R.tolist()})")
    if abs(det - 1.0) > 1e-6:
        fail(f"det R = {det:.9g}, not +1")
    sv = fit["sv"]
    slack = 2.0 * (sv[1] + sv[2]) if fit["rank"] <= 1 else 0.0
    deficit = fit["opt"] - float(np.trace(R.T @ fit["sigma"]))
    if deficit > bound["dobj"] + slack:
        fail(f"tr(R^T Sigma) is {deficit:.6g} below the optimum {fit['opt']:.6g} (bound {bound['dobj'] + slack:.3g})")
    if fit["rank"] == 0:   # R = I is specified (pcl::umeyama's result for Sigma = 0); only the fp32 cast may differ
        eI = float(np.abs(R - np.eye(3)).max())
        if eI > 2 * U32:
            fail(f"rank 0: R is not the identity, max |R - I| = {eI:.4g}")
    if fit["rank"] >= 2:
        eR = float(np.linalg.norm(R - fit["R"]))
        eT = float(np.linalg.norm(t - fit["t"]))
        out["rR"], out["rt"] = eR / bound["dR"], eT / bound["dt"]
        if eR > bound["dR"]:
            fail(f"|R - R_ref|_F = {eR:.4g} > bound {bound['dR']:.4g}")
        if eT > bound["dt"]:
            fail(f"|t - t_ref| = {eT:.4g} > bound {bound['dt']:.4g}")
    else:
        t_want = fit["dm"] - R @ fit["sm"]
        tb = bound["ddm"] + bound["dsm"] + gamma(4) * (np.linalg.norm(fit["dm"]) + 2 * np.linalg.norm(fit["sm"])) + 2 * U32 * np.linalg.norm(t_want)
        eT = float(np.linalg.norm(t - t_want))
        out["rt"] = eT / tb
        if eT > tb:
            fail(f"|t - (dm - R sm)| = {eT:.4g} > bound {tb:.4g}")
    return out


# ---- ICP ------------------------------------------------------------------------------------------------------------
def icp_step_f64(cur, tgt, tree=None):
    """One ICP iteration in float64: nearest target of every finite source (lowest index on exact ties), the gap
    between the best and the second-best squared distances (distinct target positions), the fit and the mse."""
    cur = np.asarray(cur, f64).reshape(-1, 3)
    tgt64 = np.asarray(tgt, f64).reshape(-1, 3)
    ok = np.isfinite(cur).all(1)
    tree = tree or cKDTree(tgt64)
    k = min(2, len(tgt64))
    dist, idx = tree.query(cur[ok], k=k)
    dist, idx = dist.reshape(len(idx), k), idx.reshape(len(idx), k)
    nn = idx[:, 0]
    d1 = ((cur[ok] - tgt64[nn]) ** 2).sum(1)
    gap = np.full(len(nn), np.inf)
    if k == 2:
        d2 = ((cur[ok] - tgt64[idx[:, 1]]) ** 2).sum(1)
        same = (tgt64[idx[:, 1]] == tgt64[nn]).all(1)
        gap = np.where(same, np.inf, d2 - d1)
    src_idx = np.nonzero(ok)[0]
    fit = umeyama_f64(cur[ok], tgt64[nn], ICP_PRECISION) if len(nn) >= 3 else None
    return dict(fit=fit, nn=nn, src_idx=src_idx, d1=d1, gap=gap, mse=float(d1.mean()) if len(d1) else 0.0)


def icp_f64(src, tgt, pre=None, iters=10, transforms=None):
    """ICP in float64 for `iters` steps.  Without `transforms` it is the plain float64 chain.  With `transforms`,
    the device's (or oracle's) 4x4 results after 0, 1, .., iters iterations, every step restarts from the device's
    pose: step k is fitted on src moved by transforms[k-1], judged with `check_fit` against the device's own step
    transforms[k] transforms[k-1]^-1, and the fp32 drift of the device's points (the sequential application and the
    fp32 composition, <= 2 k gamma_4 (|x| + |t|)) enters as the input error of the fit, so nothing compounds.  A step
    whose smallest nearest-target gap is within the fp32 error of the squared distances sets `decidable` False."""
    src64 = np.asarray(src, f64).reshape(-1, 3)
    P = np.eye(4) if pre is None else np.asarray(pre, f32).astype(f64).reshape(4, 4)
    tgt64 = np.asarray(tgt, f64).reshape(-1, 3)
    tree = cKDTree(tgt64)
    F = np.eye(4)
    decidable, steps, checks = True, [], []
    for k in range(1, iters + 1):
        if transforms is not None:
            F = np.asarray(transforms[k - 1], f64).reshape(4, 4)
        M = F @ P
        cur = src64 @ M[:3, :3].T + M[:3, 3]
        xmax = float(np.nanmax(np.abs(cur))) if np.isfinite(cur).any() else 0.0
        tmax = max(float(np.abs(F[:3, 3]).max()), float(np.abs(P[:3, 3]).max()))
        err = 2.0 * (k + (pre is not None)) * gamma(4) * math.sqrt(3.0) * (xmax + tmax) if transforms is not None else 0.0
        st = icp_step_f64(cur, tgt64, tree)
        if st["fit"] is None:
            break
        gap = np.minimum(st["gap"], 1e300)
        tol = 2.0 * (2.0 * np.sqrt(st["d1"]) + np.sqrt(gap) + err) * err + 8 * U32 * (2 * st["d1"] + gap)
        if (st["gap"] <= tol).any():
            decidable = False
        st.update(bound=fit_bound(st["fit"], e_in=err), err_in=err)
        steps.append(st)
        if transforms is not None:
            G = np.asarray(transforms[k], f64).reshape(4, 4)
            T = G @ np.linalg.inv(F)
            b = dict(st["bound"])
            b["dR"] += 6 * gamma(4)
            b["dt"] += 6 * gamma(4) * (float(np.linalg.norm(F[:3, 3])) + float(np.linalg.norm(T[:3, 3])))
            checks.append(check_fit(T[:3, :3], T[:3, 3], st["fit"], b))
        else:
            T = np.eye(4)
            T[:3, :3], T[:3, 3] = st["fit"]["R"], st["fit"]["t"]
            F = T @ F
    return dict(transform=F, steps=steps, checks=checks, decidable=decidable, mse=steps[-1]["mse"] if steps else 0.0)


# ---- RANSAC ---------------------------------------------------------------------------------------------------------
class Sampler:
    """rnd() = mt19937(12345)() >> 1 through numpy's MT19937 (same recurrence and seeding), in blocks"""

    def __init__(self):
        self.bg = np.random.MT19937()
        self.bg._legacy_seeding(12345)
        self.buf, self.pos = np.empty(0, np.uint64), 0

    def next(self):
        if self.pos == len(self.buf):
            self.buf, self.pos = self.bg.random_raw(3 * 1024) >> np.uint64(1), 0
        self.pos += 1
        return int(self.buf[self.pos - 1])


def sample_dist_f64(s):
    """sample_dist_thresh in float64 and the fp32 error the device's single-pass float covariance can carry"""
    s = np.asarray(s, f64)
    n = len(s)
    w = np.linalg.eigvalsh(np.cov(s.T, bias=True))
    m = float(np.sqrt(np.maximum(w, 0.0)).sum() / 3.0)
    # E[x y] - E[x] E[y] from sequential float sums: each entry off by <= gamma_n mean(|x||y|) + a few roundings
    a = np.abs(s)
    dcov = gamma(n + 4) * float(np.linalg.norm((a.T @ a) / n + np.outer(a.mean(0), a.mean(0))))
    dm = sum(min(math.sqrt(dcov), dcov / (2.0 * math.sqrt(x))) if x > 0 else math.sqrt(dcov) for x in np.maximum(w, 0.0)) / 3.0
    dm += 4 * U32 * m
    return m * m, 2.0 * m * dm + dm * dm


def ransac_f64(src_xyz, tgt_xyz, pairs, max_iterations=2000, threshold=1500.0):
    """CorrespondenceRejectorSampleConsensus as the device runs it, every decision in float64.  Returns the kept
    pairs, the best hypothesis's fit and triple, the iterations and `decidable`: False when an isSampleGood
    comparison, an inlier decision of a hypothesis the adaptive loop visits, or the best-count comparison could go
    the other way in fp32 (the device then need not agree exactly)."""
    src_xyz = np.asarray(src_xyz, f32).reshape(-1, 3)
    tgt_xyz = np.asarray(tgt_xyz, f32).reshape(-1, 3)
    pairs = np.asarray(pairs, np.int64).reshape(-1, 2)
    n = len(pairs)
    keep_all = dict(pairs=pairs.astype(np.int32), R=np.eye(3), t=np.zeros(3), iterations=0, decidable=True, fit=None,
                    n_valid=0, why=[])
    if n < 3:
        return keep_all
    s = src_xyz[pairs[:, 0]].astype(f64)
    tg = tgt_xyz[pairs[:, 1]].astype(f64)
    sdt, dsdt = sample_dist_f64(s)
    rng = Sampler()
    shuffled = list(range(n))
    thr2 = threshold * threshold
    why = []
    k_iter, iterations, n_best, best = 1.0, 0, -2147483647, None
    n_valid = 0
    log_p = math.log(1.0 - 0.99)
    while iterations < k_iter:
        good = False
        for _ in range(1000):
            for i in range(3):
                j = i + rng.next() % (n - i)
                shuffled[i], shuffled[j] = shuffled[j], shuffled[i]
            a, b, c = shuffled[:3]
            d2 = [float(((s[p] - s[q]) ** 2).sum()) for p, q in ((a, b), (a, c), (b, c))]
            if any(abs(x - sdt) <= dsdt + 4 * U32 * x for x in d2):
                why.append(f"isSampleGood of {(a, b, c)} within fp32 of sample_dist_thresh")
            good = all(x > sdt for x in d2)
            if good:
                break
        if not good:
            break
        n_valid += 1
        tri = list(shuffled[:3])
        fit = umeyama_f64(s[tri], tg[tri], RANSAC_PRECISION)
        bnd = fit_bound(fit, u=U64, k_sum=3, t_u=U64)
        r2 = ((s @ fit["R"].T + fit["t"] - tg) ** 2).sum(1)
        r = np.sqrt(r2)
        # the device's float model is off by dR |x| + dt; rank 1: the rotation about v0 is free, so a point's
        # image may be anywhere within 2 |its offset from the line through sm along v0|
        dr = bnd["dR"] * np.linalg.norm(s, axis=1) + bnd["dt"] + gamma(8) * (np.linalg.norm(s, axis=1) + np.linalg.norm(tg, axis=1) + np.linalg.norm(fit["t"]))
        if fit["rank"] == 1:   # (rank 0: R = I on both sides)
            v0 = np.linalg.svd(fit["sigma"])[2][0]
            off = s - fit["sm"]
            dr = dr + 2.0 * np.linalg.norm(off - np.outer(off @ v0, v0), axis=1)
        near = np.abs(r2 - thr2) <= 2.0 * r * dr + dr * dr + 8 * U32 * r2
        cnt = int((r2 < thr2).sum())
        if near.any():
            why.append(f"hypothesis {iterations} {tuple(tri)}: {int(near.sum())} residuals within fp32 of the threshold")
        if cnt > n_best:
            n_best, best = cnt, dict(fit=fit, triple=tri, inliers=r2 < thr2, hyp=iterations)
            w = n_best / n
            p = min(max(1.0 - w ** 3, 2.220446049250313e-16), 1.0 - 2.220446049250313e-16)
            k_iter = log_p / math.log(p)
        iterations += 1
        if iterations > max_iterations:
            break
    if best is None:
        return dict(keep_all, n_valid=n_valid, decidable=not why, why=why)
    keep = np.nonzero(best["inliers"])[0]
    if len(keep) < 3:
        return dict(keep_all, n_valid=n_valid, decidable=not why, why=why, fit=best["fit"], triple=best["triple"])
    return dict(pairs=pairs[keep].astype(np.int32), R=best["fit"]["R"], t=best["fit"]["t"], iterations=iterations,
                decidable=not why, why=why, fit=best["fit"], triple=best["triple"], n_valid=n_valid, hyp=best["hyp"])


def check_ransac_model(T_dev, ref):
    """a device RANSAC model against the float64 fit of the same triple (double fit, fp32 cast)"""
    T = np.asarray(T_dev, f64).reshape(4, 4)
    fit = ref["fit"]
    return check_fit(T[:3, :3], T[:3, 3], fit, fit_bound(fit, u=U64, k_sum=3, t_u=U64))
