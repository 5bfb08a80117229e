"""Keypoint fitting without a GPU: the fp64 reference (tests/fit_reference.py) -- its keypoint forward against the lbs_port
route and its analytic Jacobian against central differences, on a mesh model with pose-blended landmarks and on the
synthetic full skeleton -- and the argument errors of smpl_util.fit_keypoints and tik_fit_keypoints."""
import ctypes as C

import numpy as np
import pytest
import torch

import fit_reference as FR
from oracle import lbs_port, smplx_synth
from temporal_inverse_kinematics_b200 import _lib as L
from temporal_inverse_kinematics_b200 import smpl_util as SU

NAMES = SU.keypoint_names()


def _mesh(V=37):
    a = smplx_synth.make_smplx_arrays(V, seed=V)
    return a, SU.SmplxBodyModel(a, skeleton="full", landmark_vertex_ids=[v % V for v in (3, 1, 4, 1, 5)])


def test_reference_forward_matches_lbs_port():
    a, m = _mesh(200)
    rs = np.random.RandomState(1)
    F = 5
    theta, tr = rs.standard_normal((F, 22, 3)) * 0.5, rs.standard_normal((F, 3))
    for betas in (None, rs.standard_normal(10)):
        st = FR.forward(FR.model_arrays(m), theta, FR.betas_rows(betas, F, 10), tr)
        aa = np.zeros((F, 55, 3))
        aa[:, :22] = theta
        ej, ev = lbs_port.lbs(aa, dict(a, parents=FR.PARENTS55), betas, tr)
        assert np.abs(st["points"][:, :55] - ej).max() < 1e-9
        assert np.abs(st["points"][:, 55:] - ev[:, m.landmark_vertex_ids]).max() < 1e-7   # the model's weights are fp32
    s = SU.SyntheticBodyModel(skeleton="full")
    betas = rs.standard_normal(10)
    st = FR.forward(FR.model_arrays(s), theta, FR.betas_rows(betas, F, 10), tr)
    aa = np.zeros((F, 60, 3))
    aa[:, :22] = theta
    R = FR.batch_rodrigues(aa.reshape(-1, 3)).reshape(F, 60, 3, 3)
    want = FR.forward_kinematics(R, s.rest(betas).astype(np.float64), s.parents, tr)[0]
    assert np.abs(st["points"] - want).max() < 1e-6                  # rest(betas) is fp32


@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
@pytest.mark.parametrize("betas_mode,fit_transl", [("none", False), ("shared", True), ("frame", True), ("frame", False)])
def test_reference_jacobian_matches_central_differences(kind, betas_mode, fit_transl):
    m = _mesh()[1] if kind == "mesh" else SU.SyntheticBodyModel(skeleton="full")
    ma = FR.model_arrays(m)
    rs = np.random.RandomState(len(kind) + len(betas_mode))
    F = 3
    betas = {"none": None, "shared": rs.standard_normal(10), "frame": rs.standard_normal((F, 10))}[betas_mode]
    b = FR.betas_rows(betas, F, 10)
    theta, tau = rs.standard_normal((F, 22, 3)) * 0.6, rs.standard_normal((F, 3))
    sel = SU.keypoint_indices(NAMES)                                 # every joint and landmark
    J = FR.jacobian(ma, FR.forward(ma, theta, b, tau), sel, fit_transl)
    x = np.concatenate([theta.reshape(F, 66), tau], 1)
    h = 1e-6
    for a in range(J.shape[2]):
        xp, xm = x.copy(), x.copy()
        xp[:, a] += h
        xm[:, a] -= h
        fp = FR.forward(ma, xp[:, :66], b, xp[:, 66:])["points"][:, sel].reshape(F, -1)
        fm = FR.forward(ma, xm[:, :66], b, xm[:, 66:])["points"][:, sel].reshape(F, -1)
        num = (fp - fm) / (2 * h)
        assert np.abs(J[:, :, a] - num).max() < 1e-6, a
    if kind == "mesh":                                                # the pose-blend term is part of what was checked
        ma0 = dict(ma, posedirs=None)
        J0 = FR.jacobian(ma0, FR.forward(ma, theta, b, tau), sel, fit_transl)
        assert np.abs(J0 - J).max() > 1e-3


def test_reference_schedule_never_increases_cost():
    _, m = _mesh()
    rs = np.random.RandomState(3)
    F = 4
    theta = rs.standard_normal((F, 22, 3)) * 0.3
    y = FR.forward(FR.model_arrays(m), theta, np.zeros((F, 10)), np.zeros((F, 3)))["points"][:, SU.keypoint_indices("coco")]
    init = theta + rs.standard_normal(theta.shape) * 0.1
    p0, t0, e0, e0b = FR.fit(m, y, init, n_iter=0)
    assert np.array_equal(p0, init) and np.array_equal(e0, e0b)
    p, t, ei, e = FR.fit(m, y, init, n_iter=5, prior_weight=1e-4)
    assert (e <= ei).all() and (e < 0.1 * ei).all()


def test_python_argument_errors_without_a_gpu():
    _, m = _mesh()
    y, p = torch.zeros(2, 17, 3), torch.zeros(2, 22, 3)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        SU.fit_keypoints(y, m, p)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        SU.fit_keypoints(np.zeros((2, 17, 3), np.float32), m, p)
    with pytest.raises(TypeError):
        SU.fit_keypoints(y, object(), p)
    with pytest.raises(ValueError):
        SU.fit_keypoints(y, SU.SyntheticBodyModel(skeleton="body"), p)
    with pytest.raises(ValueError):
        SU.fit_keypoints(y, m, p, select=["pelvis", "tail"])


def _fake_model(L_=5, B=10, kmax=2):
    c = L.TikKeypointModel()
    c.n_betas, c.n_landmarks, c.kmax = B, L_, kmax
    c.joint_template_dev = c.joint_dirs_dev = c.lm_template_dev = c.lm_dirs_dev = 256
    c.lm_skin_idx_dev = c.lm_skin_w_dev = 256
    if B == 0:
        c.joint_dirs_dev = c.lm_dirs_dev = None
    return c


def test_c_abi_argument_errors():
    """Host-side checks of tik_fit_keypoints (no device work is reached: pointers are never dereferenced)."""
    lib, bad = L.lib(), L._H["TIK_ERR_INVALID"]
    A, Y, P0, OUT = 1 << 20, 2 << 20, 3 << 20, 4 << 20               # disjoint fake device addresses

    def call(m=None, weights=None, wpf=0, betas=None, bpf=0, fit_transl=1, sel=(0, 55), prior=1e-3, n_iter=10, F=0,
             model=True, pose_out=OUT, transl_out=None, cost=None, target=Y, init=P0):
        s = (C.c_int32 * max(1, len(sel)))(*sel)
        return lib.tik_fit_keypoints(C.byref(m or _fake_model()) if model else None, target, weights, wpf, init, betas,
                                     bpf, None, fit_transl, s, len(sel), prior, n_iter, F, pose_out, transl_out, cost, None)
    assert call() == 0                                              # F = 0: a no-op after the checks
    assert call(model=False) == bad
    assert call(_fake_model(B=17)) == bad
    assert call(_fake_model(L_=9)) == bad
    assert call(_fake_model(kmax=0)) == bad
    assert call(wpf=2) == bad and call(wpf=1) == bad                # per-frame weights without weights
    assert call(bpf=2) == bad and call(bpf=1) == bad                # per-frame betas without betas
    assert call(fit_transl=2) == bad
    assert call(sel=()) == bad and call(sel=(0,) * 65) == bad
    assert call(sel=(60,)) == bad and call(sel=(-1,)) == bad
    assert b"select" in lib.tik_last_error()
    for prior in (0.0, -1e-3, float("inf"), float("nan")):
        assert call(prior=prior) == bad
    assert b"prior_weight" in lib.tik_last_error()
    assert call(n_iter=-1) == bad and call(F=-1) == bad
    assert call(F=4, target=None) == bad and call(F=4, pose_out=None) == bad
    # outputs may not overlap inputs or each other
    assert call(F=4, pose_out=Y + 4) == bad and call(F=4, pose_out=P0) == bad
    assert call(F=4, cost=OUT + 8) == bad and call(F=4, transl_out=A, weights=A) == bad
    assert b"overlap" in lib.tik_last_error()
