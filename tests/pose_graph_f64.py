"""Float64 reference of bshot_optimize_trajectory's pose graph (numpy / scipy only), and a checker for the device's answer.

Model (DESIGN §3.9): nodes [R|t], node 0 fixed; edge (a, b) with measurement Z = [R_z | t_z];
  r_t = R_a^T (t_b - t_a) - t_z,  r_phi = Log(R_z^T R_a^T R_b),  F = 1/2 sum w_t |r_t|^2 + w_r |r_phi|^2
perturbation t <- t + rho, R <- R Exp(phi).  LM as the device runs it (lambda from 1e-4, /10 on success, *10 otherwise,
every solve an iteration, the same three stop tests), with exact sparse solves (scipy.sparse.linalg.splu).

check_optimum bounds the distance of a device result to the reference optimum x*: with H* the Gauss-Newton matrix at x*
(free nodes), a point x with gradient g(x) lies within |g|_2 / lambda_min(H*) of x* to first order.  The device's claim is
its reported |g|_inf at its float64 state (<= sqrt(6 (n - 1)) times that in 2-norm), the reference's own residual gradient
adds the same way, and the cast of the returned poses to fp32 adds each entry's rounding."""
import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla


def skew(v):
    v = np.asarray(v, np.float64)
    S = np.zeros(v.shape[:-1] + (3, 3))
    S[..., 0, 1], S[..., 0, 2], S[..., 1, 2] = -v[..., 2], v[..., 1], -v[..., 0]
    S[..., 1, 0], S[..., 2, 0], S[..., 2, 1] = v[..., 2], -v[..., 1], v[..., 0]
    return S


def so3_exp(w):
    w = np.asarray(w, np.float64)
    th2 = np.sum(w * w, axis=-1)[..., None, None]
    th = np.sqrt(th2)
    small = th < 1e-4
    ths = np.where(small, 1.0, th)
    A = np.where(small, 1.0 - th2 / 6.0 + th2 * th2 / 120.0, np.sin(ths) / ths)
    B = np.where(small, 0.5 - th2 / 24.0 + th2 * th2 / 720.0, (1.0 - np.cos(ths)) / (ths * ths))
    S = skew(w)
    return np.eye(3) + A * S + B * (S @ S)


def so3_log(R):
    R = np.asarray(R, np.float64)
    c = np.clip(0.5 * (np.trace(R, axis1=-2, axis2=-1) - 1.0), -1.0, 1.0)
    th = np.arccos(c)
    v = np.stack([R[..., 2, 1] - R[..., 1, 2], R[..., 0, 2] - R[..., 2, 0], R[..., 1, 0] - R[..., 0, 1]], -1)
    small = th < 1e-4
    ths = np.where(small, 1.0, th)
    f = np.where(small, 0.5 + th * th / 12.0 + 7.0 * th ** 4 / 720.0, ths / (2.0 * np.sin(ths)))
    return f[..., None] * v   # rotation residuals near pi do not occur in these graphs


def jr_inv(w):
    w = np.asarray(w, np.float64)
    th2 = np.sum(w * w, axis=-1)[..., None, None]
    th = np.sqrt(th2)
    small = th < 1e-4
    ths = np.where(small, 1.0, th)
    C = np.where(small, 1.0 / 12.0 + th2 / 720.0 + th2 * th2 / 30240.0, 1.0 / (ths * ths) - (1.0 + np.cos(ths)) / (2.0 * ths * np.sin(ths)))
    S = skew(w)
    return np.eye(3) + 0.5 * S + C * (S @ S)


class Graph:
    """poses: (n, 4, 4) fp32 trajectory; loops: list of (from, to, T 4x4); sigmas (mm, deg) per class"""

    def __init__(self, poses, loops, odom_sigma=(20.0, 0.1), loop_sigma=(100.0, 1.0)):
        P = np.asarray(poses, np.float32).astype(np.float64)
        self.n = len(P)
        self.R0, self.t0 = P[:, :3, :3].copy(), P[:, :3, 3].copy()
        a = np.arange(self.n - 1)
        fr = [l[0] for l in loops]
        to = [l[1] for l in loops]
        self.ea = np.concatenate([a, np.asarray(fr, np.int64)]).astype(np.int64)
        self.eb = np.concatenate([a + 1, np.asarray(to, np.int64)]).astype(np.int64)
        Zl = np.asarray([np.asarray(l[2], np.float32).astype(np.float64) for l in loops]).reshape(-1, 4, 4)
        Rz_o = np.einsum("eji,ejk->eik", self.R0[:-1], self.R0[1:])
        tz_o = np.einsum("eji,ej->ei", self.R0[:-1], self.t0[1:] - self.t0[:-1])
        self.Rz = np.concatenate([Rz_o, Zl[:, :3, :3]])
        self.tz = np.concatenate([tz_o, Zl[:, :3, 3]])
        deg = np.pi / 180.0
        L = len(loops)
        self.wt = np.concatenate([np.full(self.n - 1, 1.0 / odom_sigma[0] ** 2), np.full(L, 1.0 / loop_sigma[0] ** 2)])
        self.wr = np.concatenate([np.full(self.n - 1, 1.0 / (odom_sigma[1] * deg) ** 2), np.full(L, 1.0 / (loop_sigma[1] * deg) ** 2)])
        self.n_loops = L

    def residuals(self, R, t):
        Ra, Rb = R[self.ea], R[self.eb]
        v = np.einsum("eji,ej->ei", Ra, t[self.eb] - t[self.ea])
        rt = v - self.tz
        E = np.einsum("eji,ejk->eik", self.Rz, np.einsum("eji,ejk->eik", Ra, Rb))
        return rt, so3_log(E), v

    def edge_costs(self, R, t):
        rt, rr, _ = self.residuals(R, t)
        return 0.5 * (self.wt * np.sum(rt * rt, -1) + self.wr * np.sum(rr * rr, -1))

    def jacobians(self, R, t):
        rt, rr, v = self.residuals(R, t)
        Ra, Rb = R[self.ea], R[self.eb]
        E = len(self.ea)
        Ja, Jb = np.zeros((E, 6, 6)), np.zeros((E, 6, 6))
        RaT = np.transpose(Ra, (0, 2, 1))
        Ji = jr_inv(rr)
        Ja[:, :3, :3], Jb[:, :3, :3] = -RaT, RaT
        Ja[:, :3, 3:] = skew(v)
        Ja[:, 3:, 3:] = -Ji @ np.einsum("eji,ejk->eik", Rb, Ra)
        Jb[:, 3:, 3:] = Ji
        return np.concatenate([rt, rr], -1), Ja, Jb

    def linearize(self, R, t):
        """-> cost, g (6 (n - 1)), H (sparse, free nodes 1..n-1)"""
        r, Ja, Jb = self.jacobians(R, t)
        W = np.concatenate([np.repeat(self.wt[:, None], 3, 1), np.repeat(self.wr[:, None], 3, 1)], 1)
        F = 0.5 * np.sum(W * r * r)
        m = 6 * (self.n - 1)
        g = np.zeros(6 * self.n)
        rows, cols, vals = [], [], []
        blocks = {"aa": np.einsum("eki,ek,ekj->eij", Ja, W, Ja), "ab": np.einsum("eki,ek,ekj->eij", Ja, W, Jb), "bb": np.einsum("eki,ek,ekj->eij", Jb, W, Jb)}
        np.add.at(g, (6 * self.ea[:, None] + np.arange(6)), np.einsum("eki,ek,ek->ei", Ja, W, r))
        np.add.at(g, (6 * self.eb[:, None] + np.arange(6)), np.einsum("eki,ek,ek->ei", Jb, W, r))
        ii, jj = np.meshgrid(np.arange(6), np.arange(6), indexing="ij")
        for (ni, nj, B) in ((self.ea, self.ea, blocks["aa"]), (self.ea, self.eb, blocks["ab"]), (self.eb, self.eb, blocks["bb"]),
                            (self.eb, self.ea, np.transpose(blocks["ab"], (0, 2, 1)))):
            keep = (ni > 0) & (nj > 0)
            rows.append((6 * (ni[keep] - 1))[:, None, None] + ii)
            cols.append((6 * (nj[keep] - 1))[:, None, None] + jj)
            vals.append(B[keep])
        H = sp.csc_matrix((np.concatenate([v.ravel() for v in vals]), (np.concatenate([r_.ravel() for r_ in rows]), np.concatenate([c.ravel() for c in cols]))),
                          shape=(m, m))
        return F, g[6:], H

    def retract(self, R, t, d):
        d = d.reshape(-1, 6)
        R2, t2 = R.copy(), t.copy()
        R2[1:] = R[1:] @ so3_exp(d[:, 3:])
        t2[1:] = t[1:] + d[:, :3]
        return R2, t2

    def solve(self, max_iterations=50, grad_tolerance=1e-6, step_tolerance=1e-9):
        R, t = self.R0.copy(), self.t0.copy()
        F, g, H = self.linearize(R, t)
        lam, it, status = 1e-4, 0, 3
        while True:
            if np.abs(g).max(initial=0.0) <= grad_tolerance:
                status = 1
                break
            if it >= max_iterations:
                break
            it += 1
            A = (H + lam * sp.diags(H.diagonal())).tocsc()
            d = spla.splu(A).solve(-g)
            if np.abs(d).max() <= step_tolerance:
                status = 2
                break
            R2, t2 = self.retract(R, t, d)
            F2 = np.sum(self.edge_costs(R2, t2))
            if F2 < F:
                R, t = R2, t2
                F, g, H = self.linearize(R, t)
                lam /= 10.0
            else:
                lam *= 10.0
        return dict(R=R, t=t, cost=F, g=g, H=H, iterations=it, status=status)


def tangent_distance(R_ref, t_ref, poses):
    """per free node (t - t*, Log(R*^T R)) of fp32 poses against the reference, stacked"""
    P = np.asarray(poses, np.float32).astype(np.float64)
    dt = P[1:, :3, 3] - t_ref[1:]
    dr = so3_log(np.einsum("eji,ejk->eik", R_ref[1:], P[1:, :3, :3]))
    return np.concatenate([dt, dr], 1).ravel()


def check_optimum(graph, ref, poses, g_claim_inf, slack=1.5):
    """raises AssertionError when the fp32 poses lie farther from the reference optimum than the device's gradient claim
    allows; returns (distance, bound)"""
    m = 6 * (graph.n - 1)
    if m == 0:
        return 0.0, 0.0
    H = ref["H"]
    if m <= 600:
        lmin = float(np.linalg.eigvalsh(H.toarray())[0])
    else:
        lmin = float(spla.eigsh(H, k=1, sigma=0, which="LM", return_eigenvectors=False)[0])
    P = np.asarray(poses, np.float32)
    u = 2.0 ** -24
    rnd_t = np.sqrt(np.sum((np.abs(P[1:, :3, 3]).astype(np.float64) * u) ** 2))
    rnd_r = np.sqrt(3.0 * (graph.n - 1)) * 4.0 * u
    g_ref = float(np.linalg.norm(ref["g"]))
    bound = slack * (np.sqrt(m) * g_claim_inf + g_ref) / lmin
    d = tangent_distance(ref["R"], ref["t"], poses).reshape(-1, 6)
    dt, dr = float(np.linalg.norm(d[:, :3])), float(np.linalg.norm(d[:, 3:]))
    assert dt <= bound + 2.0 * rnd_t, f"translations {dt:.3g} mm from the reference optimum > bound {bound + 2.0 * rnd_t:.3g} (lambda_min {lmin:.3g})"
    assert dr <= bound + 2.0 * rnd_r, f"rotations {dr:.3g} rad from the reference optimum > bound {bound + 2.0 * rnd_r:.3g} (lambda_min {lmin:.3g})"
    return max(dt, dr), bound
