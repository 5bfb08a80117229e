"""tik_body_keypoints beyond the shapes smpl_util's models produce: 0 to 16 shape directions and 1 to 8 landmarks, which
select the other kernel instantiations (posedirs rows held: 16 for L <= 5, 24 for L <= 8; betas held: 0, 10 or 16),
against an fp64 oracle built from oracle/lbs_port.py pieces; and the same-device check of smpl_util.keypoints."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import lbs_port, smplx_synth
from oracle.fk_port import forward_kinematics
from oracle.geometry_port import batch_rodrigues
from temporal_inverse_kinematics_b200 import _lib as L
from temporal_inverse_kinematics_b200 import smpl_util as SU

PARENTS55 = smplx_synth.PARENTS55
TOL = 1e-4


def _pack(a, ids, B, with_posedirs):
    sd = np.asarray(a["shapedirs"], dtype=np.float64)[..., :B]
    W = np.asarray(a["weights"])[ids]
    kmax = max(1, int((W != 0).sum(1).max()))
    idx, w = np.zeros((len(ids), kmax), np.int32), np.zeros((len(ids), kmax))
    for l in range(len(ids)):
        j = np.flatnonzero(W[l])
        idx[l, :len(j)], w[l, :len(j)] = j, W[l, j]
    pd = np.asarray(a["posedirs"])[ids].reshape(3 * len(ids), -1) if with_posedirs else None
    return SU.KeypointPack(torch.device("cuda"), a["J_regressor"] @ a["v_template"], np.einsum("jv,vck->jck", a["J_regressor"], sd),
                           np.asarray(a["v_template"])[ids], sd[ids], pd, idx, w)


def _oracle(aa, a, ids, b, transl, with_posedirs):
    """fp64 points (F, 55 + L, 3): joints, then the landmark vertices `ids`; b (F, B) betas per frame."""
    F, B = b.shape
    sd = np.asarray(a["shapedirs"], dtype=np.float64)[..., :B]
    jt = lbs_port.shape(a["v_template"], sd, a["J_regressor"])[1]
    rest = jt[None] + np.einsum("jck,fk->fjc", np.einsum("jv,vck->jck", a["J_regressor"], sd), b)
    R = batch_rodrigues(np.asarray(aa, dtype=np.float64).reshape(-1, 3)).reshape(F, 55, 3, 3)
    joints, gR = forward_kinematics(R, rest, PARENTS55)
    A = np.concatenate([gR, (joints - np.einsum("fjab,fjb->fja", gR, rest))[..., None]], axis=-1)
    p = np.asarray(a["v_template"], dtype=np.float64)[ids][None] + np.einsum("lck,fk->flc", sd[ids], b)
    if with_posedirs:
        p = p + lbs_port.pose_offsets(lbs_port.pose_feature(R), a["posedirs"][ids])
    T = np.einsum("lj,fjab->flab", np.asarray(a["weights"], dtype=np.float64)[ids], A)
    v = np.einsum("flab,flb->fla", T[..., :3], p) + T[..., 3]
    return np.concatenate([joints, v], axis=1) + np.asarray(transl, dtype=np.float64)[:, None]


@pytest.mark.gpu
@pytest.mark.parametrize("n_lm,B,betas_mode,with_posedirs", [
    (5, 16, "frame", True),       # 16 rows, 16 betas
    (8, 0, "none", True),         # 24 rows, no betas
    (8, 10, "shared", True),      # 24 rows, 10 betas
    (6, 16, "frame", True),       # 24 rows, 16 betas
    (7, 13, "shared", False),     # 24 rows, 13 betas zero padded to 16, rigid landmarks
    (3, 4, "frame", True),        # 16 rows, 4 betas zero padded to 10
    (1, 10, "none", True),        # betas held by the model, none given: zero betas
])
def test_kernel_variants_match_oracle(n_lm, B, betas_mode, with_posedirs):
    a = smplx_synth.make_smplx_arrays(300, seed=50 + n_lm + B)          # 16 shape directions
    ids = [int(i) for i in np.random.RandomState(n_lm).choice(300, n_lm, replace=False)]
    pack = _pack(a, ids, B, with_posedirs)
    F = 200                                                              # three whole 64-frame tiles and a tail
    rs = np.random.RandomState(B)
    aa = (rs.standard_normal((F, 55, 3)) * 0.4).astype(np.float32)
    tr = rs.standard_normal((F, 3)).astype(np.float32)
    b = np.zeros((F, B))
    betas_dev, per_frame = None, 0
    if betas_mode == "shared":
        one = rs.standard_normal(B).astype(np.float32)
        b[:] = one
        betas_dev = torch.from_numpy(one).cuda()
    elif betas_mode == "frame":
        b = rs.standard_normal((F, B)).astype(np.float32)
        betas_dev, per_frame = torch.from_numpy(b).cuda(), 1
    sel = list(range(55 + n_lm))
    pose, t = torch.from_numpy(aa).cuda(), torch.from_numpy(tr).cuda()
    out = torch.empty(F, len(sel), 3, device="cuda")
    s = (C.c_int32 * len(sel))(*sel)
    L.check(L.lib().tik_body_keypoints(C.byref(pack.c), L.ptr(pose), 55, L.ptr(betas_dev), per_frame, L.ptr(t), s, len(sel), F,
                                       L.ptr(out), L.stream_ptr()))
    want = _oracle(aa, a, ids, b.astype(np.float64), tr, with_posedirs)
    assert np.abs(out.cpu().numpy() - want).max() < TOL


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_inputs_on_another_device_are_rejected():
    m = SU.SyntheticBodyModel(skeleton="full")
    pose = torch.zeros(4, 55, 3, device="cuda:0")
    with pytest.raises(ValueError, match="device"):
        SU.keypoints(pose, m, transl=torch.zeros(4, 3, device="cuda:1"))
    with pytest.raises(ValueError, match="device"):
        SU.keypoints(pose, m, betas=torch.zeros(4, 10, device="cuda:1"))
