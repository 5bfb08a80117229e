"""Independent cross-check of ``lbs_port`` (TEST INFRASTRUCTURE), written the way ``smplx.lbs`` is: 4x4 homogeneous
transforms ``G_i = G_parent(i) @ [[R_i, J_i - J_parent(i)], [0, 1]]``, relative transforms ``G_i - [0 | G_i [J_i; 0]]``,
a dense ``W @ A`` over the flattened 4x4 matrices and homogeneous vertices, the blend shapes as explicit per-joint loops,
float64.  It takes the local rotation matrices: the two Rodrigues forms (quaternion, skew matrix) differ by ~1e-8 through
the 1e-8 added to theta, and are compared with each other on their own (fk_scipy.rodrigues_skew)."""
import numpy as np


def lbs_homogeneous(R, model, betas=None, transl=None):
    """R (F,J,3,3) local rotations -> (joints (F,J,3), vertices (F,V,3))."""
    R = np.asarray(R, dtype=np.float64)
    F, J = R.shape[:2]
    v_shaped = np.asarray(model["v_template"], dtype=np.float64).copy()
    if betas is not None:
        for k, b in enumerate(np.asarray(betas, dtype=np.float64).reshape(-1)):
            v_shaped += b * np.asarray(model["shapedirs"], dtype=np.float64)[:, :, k]
    V = v_shaped.shape[0]
    Jr = np.asarray(model["J_regressor"], dtype=np.float64) @ v_shaped
    pd = np.asarray(model["posedirs"], dtype=np.float64)
    v_posed = np.repeat(v_shaped[None], F, axis=0)
    for j in range(1, J):                                       # pose blend shapes joint by joint
        d = R[:, j] - np.eye(3)
        for a in range(3):
            for b in range(3):
                v_posed += d[:, a, b][:, None, None] * pd[None, :, :, 9 * (j - 1) + 3 * a + b]
    G = np.zeros((F, J, 4, 4))
    for i, p in enumerate(model["parents"]):
        T = np.zeros((F, 4, 4))
        T[:, :3, :3] = R[:, i]
        T[:, :3, 3] = Jr[i] if p < 0 else Jr[i] - Jr[p]
        T[:, 3, 3] = 1.0
        G[:, i] = T if p < 0 else G[:, p] @ T
    joints = G[:, :, :3, 3].copy()
    Jh = np.concatenate([Jr, np.zeros((J, 1))], axis=1)         # [J_i; 0]
    rel = G.copy()
    rel[:, :, :, 3] -= np.einsum("fjab,jb->fja", G, Jh)
    W = np.asarray(model["weights"], dtype=np.float64)
    T = (W @ rel.reshape(F, J, 16)).reshape(F, V, 4, 4)
    vh = np.concatenate([v_posed, np.ones((F, V, 1))], axis=2)
    verts = np.einsum("fvab,fvb->fva", T, vh)[..., :3]
    if transl is not None:
        tr = np.asarray(transl, dtype=np.float64)[:, None, :]
        joints, verts = joints + tr, verts + tr
    return joints, verts
