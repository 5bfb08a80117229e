"""fp64 restatement of keypoint fitting (``smpl_util.fit_keypoints`` / ``tik_fit_keypoints``) for the tests: its own
keypoint forward built from oracle.fk_port / oracle.lbs_port, the analytic Jacobian and the Levenberg-Marquardt schedule.

Per frame, theta (22,3) axis-angle of joints 0..21 (22..54 identity), tau (3):

    E(theta, tau) = sum_k w_k |kp_k(theta, beta, tau) - y_k|^2 + lam |theta - theta0|^2

    joint point k, proper ancestor j:  d kp_k / d theta_j = -[t_k - t_j]x Rg_j Jr(theta_j)
    landmark l, joint j:               sum_{m: j anc-or-self of m} w_lm (-[x_lm - t_j]x Rg_j Jr(theta_j))
                                       + (sum_m w_lm Rg_m) d offset_l / d theta_j,
                                       d offset_l / d theta_j,a = posedirs_l[:, 9(j-1) + e] . (R_j [Jr(theta_j) e_a]x)[e]
    d kp / d tau = I

    LM: mu = 1e-3; H = J^T W J + lam I_pose, g = J^T W r + lam (theta - theta0); (H + mu diag H) delta = -g by Cholesky;
    accept iff E strictly drops (mu = max(mu/10, 1e-7)), else mu = min(mu*10, 1e7); a failed Cholesky is a rejection.
"""
import numpy as np

from oracle import lbs_port
from oracle.fk_port import forward_kinematics
from oracle.geometry_port import batch_rodrigues
from temporal_inverse_kinematics_b200 import smpl_util as SU

J55 = 55
PARENTS55 = list(SU.SMPLX_FULL_PARENTS[:J55])
ANC = []                                                 # ancestors-or-self of each joint
for _j, _p in enumerate(PARENTS55):
    ANC.append((set() if _p < 0 else set(ANC[_p])) | {_j})


def model_arrays(model):
    """The model as the keypoint kernel reads it, in fp64: jt (55,3), jd (55,3,B), lm_t (L,3), lm_d (L,3,B), posedirs
    (L,3,486) or None, dense skinning weights W (L,55)."""
    if isinstance(model, SU.SmplxBodyModel):
        ids = model.landmark_vertex_ids
        sd = model.shapedirs[..., :SU.SMPLX_NUM_BETAS]
        return dict(jt=model.J_regressor @ model.v_template, jd=np.einsum("jv,vck->jck", model.J_regressor, sd),
                    lm_t=model.v_template[ids], lm_d=sd[ids], posedirs=model.posedirs[ids].astype(np.float64),
                    W=model.weights[ids].astype(np.float64))
    L = len(SU.SMPLX_LANDMARK_NAMES)
    W = np.zeros((L, J55))
    W[:, SU.SMPLX_LANDMARK_PARENT] = 1
    rj, sd = model.rest_joints.astype(np.float64), model.joint_shapedirs.astype(np.float64)
    return dict(jt=rj[:J55], jd=sd[:J55], lm_t=rj[J55:], lm_d=sd[J55:], posedirs=None, W=W)


def betas_rows(betas, F, B):
    """None, a vector (every frame) or (F, <= B) rows -> (F, B) float64."""
    b = np.zeros((F, B))
    if betas is not None:
        v = np.asarray(betas, dtype=np.float64)
        if v.ndim == 2:
            b[:, :v.shape[1]] = v
        else:
            b[:, :v.shape[0]] = v
    return b


def forward(m, theta, betas, tau):
    """theta (F,22,3), betas (F,B), tau (F,3) -> state dict; state['points'] (F, 55 + L, 3) are the keypoints of every
    point index."""
    theta = np.array(theta, dtype=np.float64).reshape(-1, 22, 3)
    F = theta.shape[0]
    aa = np.zeros((F, J55, 3))
    aa[:, :22] = theta
    R = batch_rodrigues(aa.reshape(-1, 3)).reshape(F, J55, 3, 3)
    rest = m["jt"][None] + np.einsum("jck,fk->fjc", m["jd"], betas)
    t, gR = forward_kinematics(R, rest, PARENTS55)
    p = m["lm_t"][None] + np.einsum("lck,fk->flc", m["lm_d"], betas)
    if m["posedirs"] is not None:
        p = p + lbs_port.pose_offsets(lbs_port.pose_feature(R), m["posedirs"])
    x = np.einsum("fmab,flmb->flma", gR, p[:, :, None, :] - rest[:, None]) + t[:, None]       # (F, L, 55, 3)
    v = np.einsum("lm,flma->fla", m["W"], x)
    pts = np.concatenate([t, v], axis=1) + np.asarray(tau, dtype=np.float64)[:, None]
    return dict(theta=theta, R=R, gR=gR, t=t, rest=rest, p=p, x=x, points=pts)


def skew(v):
    v = np.asarray(v)
    z = np.zeros(v.shape[:-1])
    return np.stack([np.stack([z, -v[..., 2], v[..., 1]], -1), np.stack([v[..., 2], z, -v[..., 0]], -1),
                     np.stack([-v[..., 1], v[..., 0], z], -1)], -2)


def right_jacobian(theta):
    """(..., 3) -> (..., 3, 3): Jr = I - (1 - cos phi)/phi^2 [theta]x + (phi - sin phi)/phi^3 [theta]x^2."""
    th = np.asarray(theta, dtype=np.float64)
    phi2 = (th * th).sum(-1)[..., None, None]
    phi = np.sqrt(phi2)
    small = phi2 < 1e-6
    safe = np.where(small, 1.0, phi)
    a = np.where(small, 0.5 - phi2 / 24, (1 - np.cos(safe)) / safe ** 2)
    b = np.where(small, 1 / 6 - phi2 / 120, (safe - np.sin(safe)) / safe ** 3)
    K = skew(th)
    return np.eye(3) - a * K + b * (K @ K)


def jacobian(m, st, sel, fit_transl):
    """(F, 3n, 66 [+3]) analytic Jacobian of the selected points at the state ``st``."""
    F = st["t"].shape[0]
    n, P = len(sel), 69 if fit_transl else 66
    Jr = right_jacobian(st["theta"])                                   # (F,22,3,3)
    M = st["gR"][:, :22] @ Jr
    J = np.zeros((F, 3 * n, P))
    for k, q in enumerate(sel):
        for j in range(22):
            if q < J55:
                if j == q or j not in ANC[q]:
                    continue
                blk = -skew(st["t"][:, q] - st["t"][:, j]) @ M[:, j]
            else:
                l = q - J55
                s = np.zeros((F, 3))
                for mm in range(J55):
                    if m["W"][l, mm] != 0 and j in ANC[mm]:
                        s += m["W"][l, mm] * (st["x"][:, l, mm] - st["t"][:, j])
                blk = -skew(s) @ M[:, j]
                if m["posedirs"] is not None and j >= 1:
                    A = np.einsum("m,fmab->fab", m["W"][l], st["gR"])
                    pd = m["posedirs"][l][:, 9 * (j - 1):9 * j]             # (3, 9)
                    dR = np.stack([st["R"][:, j] @ skew(Jr[:, j, :, a]) for a in range(3)], -1)   # (F,3,3,a)
                    dp = np.einsum("ce,fea->fca", pd, dR.reshape(F, 9, 3))
                    blk = blk + A @ dp
            J[:, 3 * k:3 * k + 3, 3 * j:3 * j + 3] = blk
        if fit_transl:
            J[:, 3 * k:3 * k + 3, 66:69] = np.eye(3)
    return J


def cost(st, sel, target, w, theta0, lam):
    r = st["points"][:, sel] - target
    return (w * (r * r).sum(-1)).sum(-1) + lam * ((st["theta"] - theta0) ** 2).sum((1, 2))


def fit(model, target, init_pose, betas=None, transl=None, select="coco", weights=None, prior_weight=1e-3, n_iter=10,
        fit_transl=True):
    """The LM schedule of tik_fit_keypoints in fp64 -> (poses (F,22,3), transl (F,3), cost_init (F,), cost (F,))."""
    m = model_arrays(model)
    sel = SU.keypoint_indices(select)
    y = np.asarray(target, dtype=np.float64)
    F, n = y.shape[0], len(sel)
    theta0 = np.asarray(init_pose, dtype=np.float64).reshape(F, 22, 3)
    b = betas_rows(betas, F, m["jd"].shape[2])
    tau = np.zeros((F, 3)) if transl is None else np.asarray(transl, dtype=np.float64).copy()
    w = np.broadcast_to(np.ones(n) if weights is None else np.asarray(weights, dtype=np.float64), (F, n))
    P, lam = (69 if fit_transl else 66), prior_weight
    x = np.concatenate([theta0.reshape(F, 66), tau], 1)

    def state(xv):
        return forward(m, xv[:, :66], b, xv[:, 66:])

    st = state(x)
    E0 = cost(st, sel, y, w, theta0, lam)
    E = E0.copy()
    mu = np.full(F, 1e-3)
    live = np.isfinite(E0)
    wr = np.repeat(w, 3, axis=1)
    for _ in range(n_iter):
        J = jacobian(m, st, sel, fit_transl)
        r = (st["points"][:, sel] - y).reshape(F, -1)
        H = np.einsum("fra,fr,frb->fab", J, wr, J)
        H[:, np.arange(66), np.arange(66)] += lam
        g = np.einsum("fra,fr,fr->fa", J, wr, r)
        g[:, :66] += lam * (x[:, :66] - theta0.reshape(F, 66))
        xc = x.copy()
        ok = np.zeros(F, bool)
        for f in np.flatnonzero(live):
            A = H[f] + mu[f] * np.diag(np.diag(H[f]))
            try:
                Lc = np.linalg.cholesky(A)
            except np.linalg.LinAlgError:
                continue
            d = -np.linalg.solve(Lc.T, np.linalg.solve(Lc, g[f]))
            xc[f, :P] += d
            ok[f] = True
        stc = state(xc)
        Ec = cost(stc, sel, y, w, theta0, lam)
        acc = ok & (Ec < E)
        mu = np.where(acc, np.maximum(mu / 10, 1e-7), np.minimum(mu * 10, 1e7))
        x[acc], E[acc] = xc[acc], Ec[acc]
        for key in st:
            st[key][acc] = stc[key][acc]
    E = np.where(live, E, np.nan)
    return x[:, :66].reshape(F, 22, 3), x[:, 66:], E0, E
