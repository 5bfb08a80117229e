"""CPU linear blend skinning from the published SMPL-X formulation (TEST INFRASTRUCTURE).

**parity unpinned**, like ``fk_port``: the reference's ``run_smpl_inference(return_mesh=True)`` (common/smpl_util.py:22-82)
calls the third-party ``smplx.lbs.lbs``, which is neither vendored nor version-pinned.  This restates it in float64:

    v_shaped   = v_template + shapedirs[..., :B] . betas               (blend_shapes)
    J          = J_regressor . v_shaped                                 (vertices2joints)
    feature    = (R[1:] - I).flatten()                                  (54 x 9 = 486, row-major per joint)
    v_posed    = v_shaped + (feature . posedirs.reshape(-1, 486).T).reshape(V, 3)
    G_j, t_j   = batch_rigid_transform chain (fk_port.forward_kinematics, rest joints J)
    A_j        = [G_j | t_j - G_j J_j]                                  (relative transforms)
    T_v        = sum_j weights[v, j] A_j                                (dense W . A)
    vertex v   = T_v [v_posed_v; 1] + transl,   joints = t_j + transl

Rotations come from the quaternion Rodrigues of common/geometry.py:22-65, as in ``fk_port``.
"""
import numpy as np

from .fk_port import forward_kinematics
from .geometry_port import batch_rodrigues


def shape(v_template, shapedirs, J_regressor, betas=None):
    """-> (v_shaped (V,3), rest joints (J,3)), float64."""
    v = np.asarray(v_template, dtype=np.float64)
    if betas is not None:
        b = np.asarray(betas, dtype=np.float64).reshape(-1)
        v = v + np.einsum("vck,k->vc", np.asarray(shapedirs, dtype=np.float64)[..., :b.shape[0]], b)
    return v, np.asarray(J_regressor, dtype=np.float64) @ v


def pose_feature(rotmats):
    """(F,J,3,3) local rotations -> (F, 9 (J-1)) smplx pose feature."""
    R = np.asarray(rotmats)
    return (R[:, 1:] - np.eye(3)).reshape(R.shape[0], -1)


def pose_offsets(feature, posedirs):
    """(F,486) feature, (V,3,486) posedirs -> (F,V,3)."""
    pd = np.asarray(posedirs, dtype=np.float64)
    V = pd.shape[0]
    return (feature @ pd.reshape(V * 3, -1).T).reshape(-1, V, 3)


def relative_transforms(global_R, joints, rest_joints):
    """(F,J,3,3), (F,J,3), (J,3) -> A (F,J,3,4) = [G | t - G rest]."""
    t = joints - np.einsum("fjab,jb->fja", global_R, rest_joints)
    return np.concatenate([global_R, t[..., None]], axis=-1)


def lbs(aa, model, betas=None, transl=None, chunk=64):
    """aa (F,J,3) axis-angle; model: dict with v_template, shapedirs, posedirs, J_regressor, weights, parents.
    Returns (joints (F,J,3), vertices (F,V,3)), float64."""
    aa = np.asarray(aa, dtype=np.float64)
    F, J = aa.shape[:2]
    v_shaped, rest = shape(model["v_template"], model["shapedirs"], model["J_regressor"], betas)
    R = batch_rodrigues(aa.reshape(-1, 3)).reshape(F, J, 3, 3)
    joints, gR = forward_kinematics(R, rest, model["parents"])
    A = relative_transforms(gR, joints, rest).reshape(F, J, 12)
    W = np.asarray(model["weights"], dtype=np.float64)
    feat = pose_feature(R)
    V = v_shaped.shape[0]
    verts = np.empty((F, V, 3))
    for f0 in range(0, F, chunk):                       # (chunk, V, 12) at a time: W . A is dense over all joints
        sl = slice(f0, min(F, f0 + chunk))
        vp = v_shaped[None] + pose_offsets(feat[sl], model["posedirs"])
        T = np.matmul(W[None], A[sl]).reshape(-1, V, 3, 4)
        verts[sl] = np.einsum("fvab,fvb->fva", T[..., :3], vp) + T[..., 3]
    if transl is not None:
        tr = np.asarray(transl, dtype=np.float64)[:, None, :]
        joints, verts = joints + tr, verts + tr
    return joints, verts
