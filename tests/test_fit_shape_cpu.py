"""Shape fitting without a GPU: the fp64 reference of tests/fit_shape_reference.py -- its beta Jacobian against central
differences on a mesh model and on the synthetic full skeleton, its dense and Schur solves against each other, its
schedule's monotone cost -- and the argument errors of smpl_util.fit_keypoints_shape and tik_fit_keypoints_shape."""
import ctypes as C

import numpy as np
import pytest
import torch

import fit_reference as FR
import fit_shape_reference as FS
from oracle import smplx_synth
from temporal_inverse_kinematics_b200 import _lib as L
from temporal_inverse_kinematics_b200 import smpl_util as SU


def _model(kind):
    if kind == "mesh":
        a = smplx_synth.make_smplx_arrays(37, seed=37)
        return SU.SmplxBodyModel(a, skeleton="full", landmark_vertex_ids=[3, 1, 4, 1, 5])
    return SU.SyntheticBodyModel(skeleton="full")


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
def test_reference_beta_jacobian_matches_central_differences(kind):
    ma = FR.model_arrays(_model(kind))
    rs = np.random.RandomState(len(kind))
    F = 3
    theta, tau, beta = rs.standard_normal((F, 22, 3)) * 0.6, rs.standard_normal((F, 3)), rs.standard_normal(10)
    sel = SU.keypoint_indices(SU.keypoint_names())                    # every joint and landmark
    Jb = FS.beta_jacobian(ma, FR.forward(ma, theta, np.repeat(beta[None], F, 0), tau), sel)
    h = 1e-6
    for b in range(10):
        bp, bm = beta.copy(), beta.copy()
        bp[b] += h
        bm[b] -= h
        fp = FR.forward(ma, theta, np.repeat(bp[None], F, 0), tau)["points"][:, sel].reshape(F, -1)
        fm = FR.forward(ma, theta, np.repeat(bm[None], F, 0), tau)["points"][:, sel].reshape(F, -1)
        assert np.abs(Jb[:, :, b] - (fp - fm) / (2 * h)).max() < 1e-8, b
    assert np.abs(Jb).max() > 1e-2                                    # the shape moves the points


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
@pytest.mark.parametrize("F,fit_transl", [(1, True), (5, False), (9, True)])
def test_dense_and_schur_solves_agree(kind, F, fit_transl):
    rs = np.random.RandomState(F + len(kind))
    m = _model(kind)
    ma = FR.model_arrays(m)
    theta, beta = rs.standard_normal((F, 22, 3)) * 0.4, rs.standard_normal(10)
    y = FR.forward(ma, theta, np.repeat(beta[None], F, 0), rs.standard_normal((F, 3)))["points"][:, SU.keypoint_indices("coco")]
    init = theta + rs.standard_normal(theta.shape) * 0.1
    pr = FS.Problem(m, y, init, rs.uniform(0.5, 2, (F, 17)), "coco", 1e-2, 1e-2, fit_transl)
    x = np.concatenate([init.reshape(F, 66), rs.standard_normal((F, 3)) * 0.1], 1)
    b0 = rs.standard_normal(10) * 0.3
    blocks = pr.blocks(pr.state(x, b0), x, b0)
    for mu in (1e-3, 1.0):
        dx1, db1 = FS.solve_dense(*blocks, mu)
        dx2, db2 = FS.solve_schur(*blocks, mu)
        scale = max(np.abs(dx1).max(), np.abs(db1).max())
        assert np.abs(dx1 - dx2).max() <= 1e-9 * scale and np.abs(db1 - db2).max() <= 1e-9 * scale


def test_reference_schedule_never_increases_cost():
    m = _model("mesh")
    ma = FR.model_arrays(m)
    rs = np.random.RandomState(3)
    lengths = [1, 4, 6]
    F = sum(lengths)
    theta, beta = rs.standard_normal((F, 22, 3)) * 0.3, rs.standard_normal(10)
    y = FR.forward(ma, theta, np.repeat(beta[None], F, 0), np.zeros((F, 3)))["points"][:, SU.keypoint_indices("coco")]
    init = theta + rs.standard_normal(theta.shape) * 0.1
    p0, t0, b0, e0, e0b = FS.fit_shape(m, y, init, lengths, n_iter=0)
    assert np.array_equal(p0, init) and np.array_equal(e0, e0b) and not b0.any()
    for solver in ("dense", "schur"):
        p, t, b, ei, e = FS.fit_shape(m, y, init, lengths, n_iter=6, prior_weight=1e-4, shape_prior_weight=1e-4,
                                      solver=solver)
        assert (e <= ei).all() and (e < 0.1 * ei).all()


def test_python_argument_errors_without_a_gpu():
    m = _model("mesh")
    y, p = torch.zeros(2, 17, 3), torch.zeros(2, 22, 3)
    with pytest.raises(RuntimeError, match="fit_keypoints_shape: target must be a CUDA tensor"):
        SU.fit_keypoints_shape(y, m, p)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        SU.fit_keypoints_shape(np.zeros((2, 17, 3), np.float32), m, p)
    with pytest.raises(TypeError, match="fit_keypoints_shape needs"):
        SU.fit_keypoints_shape(y, object(), p)
    with pytest.raises(ValueError):
        SU.fit_keypoints_shape(y, SU.SyntheticBodyModel(skeleton="body"), p)
    with pytest.raises(ValueError):
        SU.fit_keypoints_shape(y, m, p, select=["pelvis", "tail"])


def _fake_model(B=10, L_=5, kmax=2):
    c = L.TikKeypointModel()
    c.n_betas, c.n_landmarks, c.kmax = B, L_, kmax
    c.joint_template_dev = c.joint_dirs_dev = c.lm_template_dev = c.lm_dirs_dev = 256
    c.lm_skin_idx_dev = c.lm_skin_w_dev = 256
    if B == 0:
        c.joint_dirs_dev = c.lm_dirs_dev = None
    return c


def test_c_abi_argument_errors():
    """Host-side checks of tik_fit_keypoints_shape and its workspace query; no device work is reached (the fake
    device addresses are never dereferenced)."""
    lib, bad = L.lib(), L._H["TIK_ERR_INVALID"]
    Y, P0, FS_, OUT, BO, WS = 1 << 20, 2 << 20, 3 << 20, 4 << 20, 5 << 20, 1 << 30
    F, S = 4, 2
    need = C.c_int64()
    assert lib.tik_fit_keypoints_shape_workspace_bytes(C.byref(_fake_model()), 17, 1, F, S, C.byref(need)) == 0
    assert need.value > 10000 * F
    z = C.c_int64(-1)
    assert lib.tik_fit_keypoints_shape_workspace_bytes(C.byref(_fake_model()), 17, 1, 0, 0, C.byref(z)) == 0 and z.value == 0
    for args in ((17, 1, F, 0), (17, 1, F, F + 1), (17, 1, F, -1), (17, 1, 0, 1), (0, 1, F, S), (17, 2, F, S)):
        assert lib.tik_fit_keypoints_shape_workspace_bytes(C.byref(_fake_model()), *args, C.byref(z)) == bad, args
    assert lib.tik_fit_keypoints_shape_workspace_bytes(C.byref(_fake_model(B=0)), 17, 1, F, S, C.byref(z)) == bad

    def call(m=None, model=True, weights=None, wpf=0, fit_transl=1, fs=FS_, n_seqs=S, betas=None, lb=1e-3, sel=(0, 55),
             prior=1e-3, n_iter=10, F=F, ws=WS, ws_bytes=None, pose_out=OUT, transl_out=None, betas_out=BO, cost=None,
             target=Y, init=P0):
        s = (C.c_int32 * max(1, len(sel)))(*sel)
        return lib.tik_fit_keypoints_shape(C.byref(m or _fake_model()) if model else None, target, weights, wpf, init, None,
                                           fit_transl, fs, n_seqs, betas, lb, s, len(sel), prior, n_iter, F, ws,
                                           need.value if ws_bytes is None else ws_bytes, pose_out, transl_out, betas_out,
                                           cost, None)
    assert call(F=0, n_seqs=0) == 0                                   # F = 0: a no-op after the checks
    assert call(model=False) == bad and call(_fake_model(B=0)) == bad and call(_fake_model(B=17)) == bad
    assert call(wpf=1) == bad and call(fit_transl=2) == bad and call(sel=()) == bad and call(sel=(60,)) == bad
    for lb in (0.0, -1.0, float("inf"), float("nan")):
        assert call(lb=lb) == bad
    assert b"shape_prior_weight" in lib.tik_last_error()
    assert call(prior=0.0) == bad and call(n_iter=-1) == bad
    for n in (0, -1, F + 1):                                          # bad n_seqs
        assert call(n_seqs=n) == bad
    assert b"n_seqs" in lib.tik_last_error()
    assert call(F=0, n_seqs=1) == bad
    assert call(ws_bytes=need.value - 1) == bad                       # workspace too small
    assert b"workspace" in lib.tik_last_error()
    assert call(ws=WS + 16) == bad                                    # not 256-byte aligned
    for kw in (dict(target=None), dict(init=None), dict(fs=None), dict(pose_out=None), dict(betas_out=None), dict(ws=None)):
        assert call(**kw) == bad, kw
    assert b"null" in lib.tik_last_error()
    # outputs may not overlap inputs, the workspace or each other
    assert call(pose_out=Y + 4) == bad and call(betas_out=FS_) == bad and call(cost=OUT + 8) == bad
    assert call(betas_out=WS + 1024) == bad and call(transl_out=BO) == bad
    assert b"overlap" in lib.tik_last_error()
