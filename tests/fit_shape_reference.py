"""fp64 restatement of the shape fit (``smpl_util.fit_keypoints_shape`` / ``tik_fit_keypoints_shape``) on top of
tests/fit_reference.py: the beta columns of the Jacobian and the per-sequence Levenberg-Marquardt schedule with two
solvers for the damped system of a sequence's unknowns (F_s poses [+ translations] and the B betas):

    dense: the whole (F_s P + B)^2 system, numpy Cholesky -- the independent check, for short sequences;
    schur: per frame Y_f = (H_f + mu D_f)^-1 [C_f | g_f], then
           (sum_f (H_bb,f - C_f^T Y_f[:, :B]) + lb I + mu diag(sum_f H_bb,f + lb I)) dbeta
               = -(sum_f (g_b,f - C_f^T Y_f[:, B]) + lb beta),
           dx_f = -(Y_f[:, B] + Y_f[:, :B] dbeta) -- the kernel's algebra, feasible for long sequences.

    beta columns:  joint point k:  dt_k/dbeta = jd_root + sum_{m on root -> k, m != root} Rg_par(m) (jd_m - jd_par(m))
                   landmark l:     dv_l/dbeta = sum_m w_lm (Rg_m (lm_d_l - jd_m) + dt_m/dbeta)
"""
import numpy as np

import fit_reference as FR
from temporal_inverse_kinematics_b200 import smpl_util as SU


def beta_jacobian(m, st, sel):
    """(F, 3n, B) derivative of the selected points with respect to beta at the state ``st`` of FR.forward."""
    gR, jd, F = st["gR"], m["jd"], st["gR"].shape[0]
    B = jd.shape[2]
    dT = np.zeros((F, FR.J55, 3, B))
    for j, par in enumerate(FR.PARENTS55):
        dT[:, j] = jd[j][None] if par < 0 else gR[:, par] @ (jd[j] - jd[par])[None] + dT[:, par]
    out = np.zeros((F, 3 * len(sel), B))
    for k, q in enumerate(sel):
        if q < FR.J55:
            out[:, 3 * k:3 * k + 3] = dT[:, q]
        else:
            l = q - FR.J55
            acc = np.zeros((F, 3, B))
            for mm in range(FR.J55):
                if m["W"][l, mm] != 0:
                    acc += m["W"][l, mm] * (gR[:, mm] @ (m["lm_d"][l] - jd[mm])[None] + dT[:, mm])
            out[:, 3 * k:3 * k + 3] = acc
    return out


class Problem:
    """One sequence's data and its cost; x (F, 69) = theta (66) | tau (3)."""

    def __init__(self, model, target, init_pose, weights, select, prior_weight, shape_prior_weight, fit_transl):
        self.m = FR.model_arrays(model)
        self.sel = SU.keypoint_indices(select)
        self.y = np.asarray(target, dtype=np.float64)
        self.F, n = self.y.shape[0], len(self.sel)
        self.theta0 = np.asarray(init_pose, dtype=np.float64).reshape(self.F, 22, 3)
        w = np.ones(n) if weights is None else np.asarray(weights, dtype=np.float64)
        self.w = np.broadcast_to(w, (self.F, n))
        self.lam, self.lb, self.fit_transl = prior_weight, shape_prior_weight, fit_transl
        self.P = 69 if fit_transl else 66
        self.B = self.m["jd"].shape[2]

    def state(self, x, beta):
        return FR.forward(self.m, x[:, :66], np.repeat(np.asarray(beta)[None], self.F, 0), x[:, 66:])

    def cost(self, st, beta):
        return FR.cost(st, self.sel, self.y, self.w, self.theta0, self.lam).sum() + self.lb * float(beta @ beta)

    def blocks(self, st, x, beta):
        """H (F,P,P), g (F,P), C (F,P,B), the summed beta block Hbb + lb I and gradient gb + lb beta."""
        F = self.F
        Jx = FR.jacobian(self.m, st, self.sel, self.fit_transl)
        Jb = beta_jacobian(self.m, st, self.sel)
        r = (st["points"][:, self.sel] - self.y).reshape(F, -1)
        wr = np.repeat(self.w, 3, axis=1)
        WJx, WJb = Jx * wr[:, :, None], Jb * wr[:, :, None]
        H = np.swapaxes(WJx, 1, 2) @ Jx
        H[:, np.arange(66), np.arange(66)] += self.lam
        g = (np.swapaxes(WJx, 1, 2) @ r[:, :, None])[:, :, 0]
        g[:, :66] += self.lam * (x[:, :66] - self.theta0.reshape(F, 66))
        C = np.swapaxes(WJx, 1, 2) @ Jb
        Hbb = (np.swapaxes(WJb, 1, 2) @ Jb).sum(0) + self.lb * np.eye(self.B)
        gb = (WJb * r[:, :, None]).sum((0, 1)) + self.lb * beta
        return H, g, C, Hbb, gb


def solve_dense(H, g, C, Hbb, gb, mu):
    """The damped system of all unknowns at once -> (dx (F,P), dbeta (B)) or None when Cholesky fails."""
    F, P = g.shape
    B = Hbb.shape[0]
    N = F * P + B
    A = np.zeros((N, N))
    for f in range(F):
        A[f * P:(f + 1) * P, f * P:(f + 1) * P] = H[f]
        A[f * P:(f + 1) * P, F * P:] = C[f]
        A[F * P:, f * P:(f + 1) * P] = C[f].T
    A[F * P:, F * P:] = Hbb
    A[np.arange(N), np.arange(N)] *= 1 + mu
    try:
        Lc = np.linalg.cholesky(A)
    except np.linalg.LinAlgError:
        return None
    d = -np.linalg.solve(Lc.T, np.linalg.solve(Lc, np.concatenate([g.reshape(-1), gb])))
    return d[:F * P].reshape(F, P), d[F * P:]


def solve_schur(H, g, C, Hbb, gb, mu):
    """The same system by the Schur complement on the betas (the kernel's algebra)."""
    F, P = g.shape
    B = Hbb.shape[0]
    A = H.copy()
    A[:, np.arange(P), np.arange(P)] *= 1 + mu
    try:
        Lc = np.linalg.cholesky(A)
    except np.linalg.LinAlgError:
        return None
    rhs = np.concatenate([C, g[:, :, None]], 2)
    Y = np.linalg.solve(np.swapaxes(Lc, 1, 2), np.linalg.solve(Lc, rhs))          # (F, P, B + 1)
    S = Hbb.copy()
    S[np.arange(B), np.arange(B)] *= 1 + mu
    S -= np.einsum("fpa,fpb->ab", C, Y[:, :, :B])
    r = gb - np.einsum("fpa,fp->a", C, Y[:, :, B])
    try:
        Ls = np.linalg.cholesky(S)
    except np.linalg.LinAlgError:
        return None
    db = -np.linalg.solve(Ls.T, np.linalg.solve(Ls, r))
    return -(Y[:, :, B] + Y[:, :, :B] @ db), db


def fit_shape(model, target, init_pose, lengths=None, betas=None, transl=None, select="coco", weights=None,
              prior_weight=1e-3, shape_prior_weight=1e-3, n_iter=10, fit_transl=True, solver="dense"):
    """The schedule of tik_fit_keypoints_shape in fp64 -> (poses (F,22,3), transl (F,3), betas (S,B), cost_init (S,),
    cost (S,)).  weights: None, (n) or (F, n); betas: None, (B') or (S, B')."""
    y = np.asarray(target, dtype=np.float64)
    F = y.shape[0]
    lengths = [F] if lengths is None else list(lengths)
    starts = np.concatenate([[0], np.cumsum(lengths)]).astype(int)
    init = np.asarray(init_pose, dtype=np.float64).reshape(F, 22, 3)
    tau = np.zeros((F, 3)) if transl is None else np.asarray(transl, dtype=np.float64)
    wts = None if weights is None else np.asarray(weights, dtype=np.float64)
    solve = solve_dense if solver == "dense" else solve_schur
    poses, tr, bout, e0s, es = [], [], [], [], []
    for s, (a, b) in enumerate(zip(starts[:-1], starts[1:])):
        w = None if wts is None else (wts[a:b] if wts.ndim == 2 else wts)
        pr = Problem(model, y[a:b], init[a:b], w, select, prior_weight, shape_prior_weight, fit_transl)
        beta = np.zeros(pr.B)
        if betas is not None:
            v = np.asarray(betas, dtype=np.float64)
            v = v[s] if v.ndim == 2 else v
            beta[:v.shape[0]] = v
        x = np.concatenate([init[a:b].reshape(-1, 66), tau[a:b]], 1)
        st = pr.state(x, beta)
        E0 = pr.cost(st, beta)
        E, mu = E0, 1e-3
        if np.isfinite(E0):
            for _ in range(n_iter):
                step = solve(*pr.blocks(st, x, beta), mu)
                if step is not None:
                    xc, bc = x.copy(), beta + step[1]
                    xc[:, :pr.P] += step[0]
                    stc = pr.state(xc, bc)
                    Ec = pr.cost(stc, bc)
                if step is not None and Ec < E:
                    x, beta, st, E = xc, bc, stc, Ec
                    mu = max(mu / 10, 1e-7)
                else:
                    mu = min(mu * 10, 1e7)
        else:
            E = np.nan
        poses.append(x[:, :66].reshape(-1, 22, 3))
        tr.append(x[:, 66:])
        bout.append(beta)
        e0s.append(E0)
        es.append(E)
    return np.concatenate(poses), np.concatenate(tr), np.stack(bout), np.array(e0s), np.array(es)
