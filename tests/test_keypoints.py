"""Body keypoints without the mesh (smpl_util.keypoints, run_smpl_keypoints, tik_body_keypoints): the model packing, the
selection, argument errors, and on the GPU the kernel against an fp64 oracle, against today's routes (lbs() and fk_body
gathered), per-frame betas, guard regions, CUDA-graph replay and the device round trip into forward_windows.

The oracle restates smplx's lbs for the joints and the landmark vertices only (oracle/lbs_port.py pieces), so that large
frame counts stay cheap; the first test pins it to lbs_port.lbs."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import lbs_port, smplx_synth
from oracle.fk_port import forward_kinematics
from oracle.geometry_port import batch_rodrigues
from temporal_inverse_kinematics_b200 import _lib as L
from temporal_inverse_kinematics_b200 import smpl_util as SU
from temporal_inverse_kinematics_b200.keypoints_util import generate_smplx_to_coco_mappings

PARENTS55 = smplx_synth.PARENTS55
PARENTS60 = PARENTS55 + [SU.SMPLX_LANDMARK_PARENT] * 5
TOL = 1e-4
NAMES = SU.keypoint_names()


def _betas_rows(betas, F, per_frame):
    b = np.zeros((F, 10))
    if betas is not None:
        v = np.asarray(betas, dtype=np.float64)
        if per_frame:
            b[:, :v.shape[1]] = v
        else:
            b[:, :v.shape[0]] = v
    return b


def _aa55(aa):
    aa = np.asarray(aa, dtype=np.float64)
    out = np.zeros((aa.shape[0], 55, 3))
    n = min(aa.shape[1], 55)
    out[:, :n] = aa[:, :n]
    return out


def oracle_mesh_points(aa, a, ids, betas=None, transl=None, per_frame=False):
    """fp64 points (F, 55 + L, 3) of an SMPL-X model file: the 55 joints then the landmark vertices `ids`, from
    lbs_port's shape / pose_feature / pose_offsets on the landmark rows, fk_port and the relative transforms."""
    aa = _aa55(aa)
    F = aa.shape[0]
    b = _betas_rows(betas, F, per_frame)
    sd = np.asarray(a["shapedirs"], dtype=np.float64)[..., :10]
    jt = lbs_port.shape(a["v_template"], a["shapedirs"], a["J_regressor"])[1]
    jd = np.einsum("jv,vck->jck", a["J_regressor"], sd)
    rest = jt[None] + np.einsum("jck,fk->fjc", jd, b)                               # (F,55,3) = lbs_port.shape per frame
    R = batch_rodrigues(aa.reshape(-1, 3)).reshape(F, 55, 3, 3)
    joints, gR = forward_kinematics(R, rest, PARENTS55)
    A = np.concatenate([gR, (joints - np.einsum("fjab,fjb->fja", gR, rest))[..., None]], axis=-1)
    p = (np.asarray(a["v_template"], dtype=np.float64)[ids][None] + np.einsum("lck,fk->flc", sd[ids], b)
         + lbs_port.pose_offsets(lbs_port.pose_feature(R), a["posedirs"][ids]))
    T = np.einsum("lj,fjab->flab", np.asarray(a["weights"], dtype=np.float64)[ids], A)
    v = np.einsum("flab,flb->fla", T[..., :3], p) + T[..., 3]
    pts = np.concatenate([joints, v], axis=1)
    if transl is not None:
        pts = pts + np.asarray(transl, dtype=np.float64)[:, None]
    return pts


def oracle_synthetic_points(aa, model, betas=None, transl=None, per_frame=False):
    """fp64 points (F, 60, 3) of a SyntheticBodyModel(skeleton='full'): FK of the 60-joint tree, rest(betas) per frame."""
    aa = _aa55(aa)
    F = aa.shape[0]
    b = _betas_rows(betas, F, per_frame)
    rest = model.rest_joints.astype(np.float64)[None] + np.einsum("jck,fk->fjc", model.joint_shapedirs.astype(np.float64), b)
    R = batch_rodrigues(np.concatenate([aa, np.zeros((F, 5, 3))], 1).reshape(-1, 3)).reshape(F, 60, 3, 3)
    return forward_kinematics(R, rest, PARENTS60, transl)[0]


_MODELS = {}


def _mesh_model(V, skeleton="full"):
    if (V, skeleton) not in _MODELS:
        a = smplx_synth.make_smplx_arrays(V, seed=V)
        lm = SU.SMPLX_LANDMARK_VERTEX_IDS if V > max(SU.SMPLX_LANDMARK_VERTEX_IDS) else [v % V for v in (3, 1, 4, 1, 5)]
        _MODELS[(V, skeleton)] = (a, SU.SmplxBodyModel(a, skeleton=skeleton, landmark_vertex_ids=lm))
    return _MODELS[(V, skeleton)]


def _finger_model():
    """Landmarks skinned to up to eight joints each, finger joints among them."""
    if "finger" not in _MODELS:
        a = smplx_synth.make_smplx_arrays(40, seed=41)
        ids = [5, 11, 17, 23, 29]
        sets = [[15, 27, 39, 52], [15, 22, 23, 24, 12, 9, 30, 45], [54], [40, 41, 42, 43, 44, 45, 46, 47], [0, 15]]
        rs = np.random.RandomState(3)
        for v, js in zip(ids, sets):
            a["weights"][v] = 0
            a["weights"][v, js] = rs.dirichlet(np.ones(len(js)))
        _MODELS["finger"] = (a, SU.SmplxBodyModel(a, skeleton="full", landmark_vertex_ids=ids))
    return _MODELS["finger"]


# ------------------------------------------------------------------ CPU


def test_oracle_helper_matches_lbs_port():
    a = smplx_synth.make_smplx_arrays(200, seed=2)
    ids = [10, 20, 30, 40, 199]
    rs = np.random.RandomState(1)
    aa, tr, betas = rs.standard_normal((6, 55, 3)) * 0.5, rs.standard_normal((6, 3)), rs.standard_normal(10)
    ej, ev = lbs_port.lbs(aa, dict(a, parents=PARENTS55), betas, tr)
    got = oracle_mesh_points(aa, a, ids, betas, tr)
    assert np.abs(got[:, :55] - ej).max() < 1e-9 and np.abs(got[:, 55:] - ev[:, ids]).max() < 1e-9
    per = rs.standard_normal((6, 10))
    got = oracle_mesh_points(aa, a, ids, per, None, per_frame=True)
    for f in range(6):
        ej, ev = lbs_port.lbs(aa[f:f + 1], dict(a, parents=PARENTS55), per[f])
        assert np.abs(got[f, :55] - ej[0]).max() < 1e-9 and np.abs(got[f, 55:] - ev[0, ids]).max() < 1e-9


def test_mesh_model_packing():
    a, m = _mesh_model(37)
    pk = m.keypoint_pack("cpu")
    jt, jd = pk.jt.double().numpy(), pk.jd.double().numpy()
    assert pk.n_betas == 10 and pk.n_landmarks == 5 and jd.shape == (55, 3, 10)
    for betas in (None, np.linspace(-1, 1, 10), np.random.RandomState(0).standard_normal(10) * 2):
        want = lbs_port.shape(a["v_template"], a["shapedirs"][..., :10], a["J_regressor"], betas)[1]
        got = jt + (0 if betas is None else jd @ betas)
        assert np.abs(got - want).max() < 1e-5
    ids = m.landmark_vertex_ids
    assert np.array_equal(pk.lm_t.numpy(), a["v_template"][ids].astype(np.float32))
    assert np.array_equal(pk.lm_d.numpy(), a["shapedirs"][ids, :, :10].astype(np.float32))
    assert np.array_equal(pk.lm_posedirs.numpy(), a["posedirs"][ids].reshape(15, 486).astype(np.float32))
    dense = np.zeros((5, 55), np.float32)
    for l in range(5):
        for k in range(pk.kmax):
            dense[l, pk.skin_idx[l, k]] += pk.skin_w[l, k].item()
    assert np.array_equal(dense, a["weights"][ids].astype(np.float32))
    # landmark ids are checked here whatever the skeleton
    body = SU.SmplxBodyModel(a, skeleton="body", landmark_vertex_ids=[0, 1, 2, 3, 40])
    with pytest.raises(ValueError, match="landmark"):
        body.keypoint_pack("cpu")


def test_synthetic_mapping_reproduces_rest():
    m = SU.SyntheticBodyModel(skeleton="full")
    pk = m.keypoint_pack("cpu")
    assert pk.lm_posedirs is None and pk.kmax == 1
    assert (pk.skin_idx == 15).all() and (pk.skin_w == 1).all()
    for betas in (None, np.linspace(-2, 2, 10)):
        b = np.zeros(10) if betas is None else betas
        got = np.concatenate([pk.jt.numpy() + pk.jd.numpy() @ b, pk.lm_t.numpy() + pk.lm_d.numpy() @ b])
        assert np.abs(got - m.rest(betas)).max() < 1e-6
    with pytest.raises(ValueError):
        SU.SyntheticBodyModel(skeleton="body").keypoint_pack("cpu")


def test_coco_selection_and_names():
    assert NAMES == SU.SMPLX_FULL_JOINT_NAMES + SU.SMPLX_LANDMARK_NAMES
    assert SU.keypoint_indices("coco") == generate_smplx_to_coco_mappings(NAMES)
    assert SU.keypoint_indices(["nose", "pelvis", "right_thumb3"]) == [55, 0, 54]
    for bad in ("all", ["pelvis", "tail"], [], ["pelvis"] * 65):
        with pytest.raises(ValueError):
            SU.keypoint_indices(bad)


def test_python_argument_errors_without_a_gpu():
    _, m = _mesh_model(37)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        SU.keypoints(torch.zeros(2, 55, 3), m)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        SU.keypoints(np.zeros((2, 55, 3), np.float32), m)
    with pytest.raises(TypeError):
        SU.keypoints(torch.zeros(2, 55, 3), object())
    with pytest.raises(ValueError):
        SU.keypoints(torch.zeros(2, 55, 3), SU.SyntheticBodyModel(skeleton="body"))
    with pytest.raises(ValueError):
        SU.keypoints(torch.zeros(2, 55, 3), m, select=["pelvis", "tail"])


def _fake_model(L_=5, B=10, kmax=2):
    c = L.TikKeypointModel()
    c.n_betas, c.n_landmarks, c.kmax = B, L_, kmax
    c.joint_template_dev = c.joint_dirs_dev = c.lm_template_dev = c.lm_dirs_dev = 256
    c.lm_skin_idx_dev = c.lm_skin_w_dev = 256
    if B == 0:
        c.joint_dirs_dev = c.lm_dirs_dev = None
    return c


def test_c_abi_argument_errors():
    """Host-side checks of tik_body_keypoints (no device work is reached: pointers are never dereferenced)."""
    lib, bad = L.lib(), L._H["TIK_ERR_INVALID"]

    def call(m=None, pose_J=55, betas=None, per_frame=0, sel=(0, 55), F=0, model=True):
        s = (C.c_int32 * max(1, len(sel)))(*sel)
        return lib.tik_body_keypoints(C.byref(m or _fake_model()) if model else None, 256, pose_J, betas, per_frame, None, s,
                                      len(sel), F, 256, None)
    assert call() == 0                                              # F = 0: a no-op after the checks
    assert call(model=False) == bad
    assert call(_fake_model(B=17)) == bad
    assert call(_fake_model(L_=9)) == bad
    assert call(_fake_model(kmax=0)) == bad
    assert call(_fake_model(kmax=56)) == bad
    m = _fake_model()
    m.joint_dirs_dev = None
    assert call(m) == bad
    for pj in (21, 23, 56, 61):
        assert call(pose_J=pj) == bad
    assert call(per_frame=2) == bad
    assert call(per_frame=1) == bad                                 # per-frame betas without betas
    assert call(sel=()) == bad and call(sel=(0,) * 65) == bad
    assert call(sel=(60,)) == bad and call(sel=(-1,)) == bad        # 55 + L = 60 points
    assert call(F=-1) == bad
    assert call(_fake_model(L_=0, B=0), sel=(54,)) == 0 and call(_fake_model(L_=0, B=0), sel=(55,)) == bad
    assert b"select" in lib.tik_last_error()


# ------------------------------------------------------------------ GPU


def _inputs(F, PJ, seed, betas_mode, with_transl):
    rs = np.random.RandomState(seed)
    aa = (rs.standard_normal((F, PJ, 3)) * 0.4).astype(np.float32)
    betas = {"none": None, "shared": rs.standard_normal(10).astype(np.float32),
             "frame": rs.standard_normal((F, 10)).astype(np.float32)}[betas_mode]
    tr = rs.standard_normal((F, 3)).astype(np.float32) if with_transl else None
    return aa, betas, tr


def _run(m, aa, betas, tr, select):
    b = torch.from_numpy(betas).cuda() if betas is not None and betas.ndim == 2 else betas
    return SU.keypoints(torch.from_numpy(aa).cuda(), m, b, None if tr is None else torch.from_numpy(tr).cuda(), select)


@pytest.mark.gpu
@pytest.mark.parametrize("V,F,betas_mode,with_transl,PJ,select", [
    (37, 1, "none", False, 55, "coco"), (37, 7, "shared", True, 22, "all"), (37, 255, "frame", True, 60, "coco"),
    (37, 257, "frame", False, 55, "all"), (37, 100003, "shared", True, 55, "coco"), (10475, 1, "frame", True, 60, "all"),
    (10475, 7, "none", True, 55, "coco"), (10475, 255, "shared", False, 22, "coco"), (10475, 257, "shared", True, 60, "all"),
    (10475, 100003, "frame", True, 55, "coco"), (10475, 100003, "none", False, 22, "all"),
])
def test_keypoints_fp32_matches_oracle(V, F, betas_mode, with_transl, PJ, select):
    a, m = _mesh_model(V)
    aa, betas, tr = _inputs(F, PJ, V + F + PJ, betas_mode, with_transl)
    sel = NAMES if select == "all" else "coco"
    got = _run(m, aa, betas, tr, sel).cpu().numpy()
    want = oracle_mesh_points(aa, a, m.landmark_vertex_ids, betas, tr, per_frame=betas_mode == "frame")
    idx = SU.keypoint_indices(sel)
    assert got.shape == (F, len(idx), 3)
    assert np.abs(got - want[:, idx]).max() < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("F,betas_mode,with_transl,PJ", [(1, "none", False, 60), (255, "shared", True, 55),
                                                         (100003, "frame", True, 22), (257, "frame", False, 60)])
def test_keypoints_synthetic_matches_oracle(F, betas_mode, with_transl, PJ):
    m = SU.SyntheticBodyModel(skeleton="full")
    aa, betas, tr = _inputs(F, PJ, F + PJ, betas_mode, with_transl)
    got = _run(m, aa, betas, tr, NAMES).cpu().numpy()
    want = oracle_synthetic_points(aa, m, betas, tr, per_frame=betas_mode == "frame")
    assert np.abs(got - want).max() < TOL


@pytest.mark.gpu
def test_finger_skinned_landmarks_and_finger_selection():
    a, m = _finger_model()
    aa, betas, tr = _inputs(300, 55, 9, "frame", True)
    sel = ["left_index3", "right_thumb3", "nose", "left_ear", "right_pinky2", "right_eye", "left_eye", "right_ear", "jaw",
           "left_wrist", "nose"]
    got = _run(m, aa, betas, tr, sel).cpu().numpy()
    want = oracle_mesh_points(aa, a, m.landmark_vertex_ids, betas, tr, per_frame=True)
    assert np.abs(got - want[:, SU.keypoint_indices(sel)]).max() < TOL
    assert np.array_equal(got[:, 2], got[:, 10])
    # a selection of landmarks only still walks every finger chain the landmarks are skinned to
    got = _run(m, aa, betas, tr, SU.SMPLX_LANDMARK_NAMES).cpu().numpy()
    assert np.abs(got - want[:, 55:]).max() < TOL


@pytest.mark.gpu
def test_keypoints_agree_with_lbs_and_fk_body():
    _, m = _mesh_model(10475)
    aa, betas, tr = _inputs(300, 55, 4, "shared", True)
    pose, transl = torch.from_numpy(aa).cuda(), torch.from_numpy(tr).cuda()
    joints, _ = SU.lbs(pose, m, betas, transl)
    coco = SU.keypoint_indices("coco")
    assert (SU.keypoints(pose, m, betas, transl) - joints[:, coco]).abs().max().item() < TOL
    s = SU.SyntheticBodyModel(skeleton="full")
    p60 = torch.cat([pose, torch.zeros(300, 5, 3, device="cuda")], 1)
    fk = SU.fk_body(p60, s.rest(betas), s.parents, transl)
    assert (SU.keypoints(pose, s, betas, transl, NAMES) - fk).abs().max().item() < TOL


@pytest.mark.gpu
def test_run_smpl_keypoints_matches_run_smpl_inference(tmp_path):
    smplx_synth.write_smplx_dir(str(tmp_path), 10475, seed=20)
    rs = np.random.RandomState(4)
    F = 90
    data = {"poses": (rs.standard_normal((F, 156)) * 0.3).astype(np.float32), "gender": "female",
            "trans": rs.standard_normal((F, 3)).astype(np.float32), "betas": rs.standard_normal(16).astype(np.float32)}
    for models in (SU.load_smplx_models(str(tmp_path), "cuda", 8, skeleton="full"), SU.load_smplx_models(None, "cuda", 8, skeleton="full")):
        names = models["female"].joint_names
        for trans, root, shape in ((True, True, True), (False, True, False), (True, False, True), (False, False, False)):
            kw = dict(apply_trans=trans, apply_root_rot=root, apply_shape=shape)
            got = SU.run_smpl_keypoints(data, models, "cuda", **kw)
            want = SU.smplx_joints_to_coco(SU.run_smpl_inference(data, models, "cuda", **kw), names)
            assert got.shape == (F, 17, 3) and got.dtype == np.float32
            assert np.abs(got - want).max() < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["mesh", "synthetic"])
def test_per_frame_betas_are_bit_identical_to_broadcast_calls(kind):
    m = _mesh_model(37)[1] if kind == "mesh" else SU.SyntheticBodyModel(skeleton="full")
    F = 130
    aa, betas, tr = _inputs(F, 55, 8, "frame", True)
    pose, transl = torch.from_numpy(aa).cuda(), torch.from_numpy(tr).cuda()
    got = SU.keypoints(pose, m, torch.from_numpy(betas).cuda(), transl, NAMES)
    for f in range(F):
        one = SU.keypoints(pose[f:f + 1], m, betas[f], transl[f:f + 1], NAMES)
        assert torch.equal(got[f:f + 1], one), f


def _raw_call(pack, pose, betas, per_frame, tr, sel, out):
    s = (C.c_int32 * len(sel))(*sel)
    return L.lib().tik_body_keypoints(C.byref(pack.c), L.ptr(pose), pose.shape[1], L.ptr(betas), per_frame, L.ptr(tr), s,
                                      len(sel), pose.shape[0], L.ptr(out), L.stream_ptr())


@pytest.mark.gpu
def test_keypoints_write_only_their_outputs():
    """Outputs carved out of sentinel-filled buffers, F around the 64-frame tile, bulk and staged (unaligned) tiles."""
    GUARD, SENT = 4096, 12345.0
    _, m = _mesh_model(10475)
    pack = m.keypoint_pack(torch.device("cuda"))
    sel = SU.keypoint_indices("coco")
    for F in (1, 63, 64, 65, 128, 129, 1000):
        for shift in (0, 1):                                         # shift = 1: out is 4-byte aligned only
            aa, betas, tr = _inputs(F, 60, F, "frame", True)
            pose, b, t = torch.from_numpy(aa).cuda(), torch.from_numpy(betas).cuda(), torch.from_numpy(tr).cuda()
            n = F * 17 * 3
            buf = torch.full((GUARD + n + GUARD + 1,), SENT, device="cuda")
            out = buf[GUARD + shift:GUARD + shift + n]
            L.check(_raw_call(pack, pose, b, 1, t, sel, out))
            torch.cuda.synchronize()
            assert bool((buf[:GUARD + shift] == SENT).all()) and bool((buf[GUARD + shift + n:] == SENT).all()), (F, shift)
            assert bool(torch.isfinite(out).all()) and not bool((out == SENT).any()), (F, shift)
            ref = SU.keypoints(pose, m, b, t)
            assert torch.equal(out.view(F, 17, 3), ref), (F, shift)


@pytest.mark.gpu
def test_zero_frames_and_cuda_graph_replay():
    _, m = _mesh_model(10475)
    z = SU.keypoints(torch.zeros(0, 55, 3, device="cuda"), m, np.ones(10), torch.zeros(0, 3, device="cuda"))
    assert z.shape == (0, 17, 3)
    pack = m.keypoint_pack(torch.device("cuda"))
    F = 1000
    aa, betas, tr = _inputs(F, 55, 11, "frame", True)
    pose, b, t = torch.from_numpy(aa).cuda(), torch.from_numpy(betas).cuda(), torch.from_numpy(tr).cuda()
    sel = list(range(60))
    eager, graphed = torch.empty(F, 60, 3, device="cuda"), torch.zeros(F, 60, 3, device="cuda")
    L.check(_raw_call(pack, pose, b, 1, t, sel, eager))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        L.check(_raw_call(pack, pose, b, 1, t, sel, graphed))
    g.replay()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(graphed, eager)


@pytest.mark.gpu
def test_shape_errors_before_launch():
    _, m = _mesh_model(37)
    p = torch.zeros(3, 55, 3, device="cuda")
    for kw in (dict(pose=torch.zeros(3, 54, 3, device="cuda")), dict(transl=torch.zeros(2, 3, device="cuda")),
               dict(betas=torch.zeros(2, 10, device="cuda")), dict(betas=torch.zeros(3, 11, device="cuda")),
               dict(betas=np.zeros(11))):
        with pytest.raises(ValueError):
            SU.keypoints(kw.pop("pose", p), m, **kw)
    with pytest.raises(RuntimeError):
        SU.keypoints(p, m, transl=torch.zeros(3, 3))
    with pytest.raises(RuntimeError):
        SU.keypoints(p, m, betas=torch.zeros(3, 10))


@pytest.mark.gpu
def test_device_round_trip_into_forward_windows():
    """keypoints -> PoseRegressor.forward_windows on the device gives the poses of the numpy route through run_inference."""
    from oracle import stgcn_port as sp, synth
    from temporal_inverse_kinematics_b200 import inference
    from temporal_inverse_kinematics_b200.keypoints_util import COCO_ROOT_PAIR
    from temporal_inverse_kinematics_b200.pose_regressor import IKPoseTrainer
    tr = IKPoseTrainer().eval()
    tr.regressor.load_state_dict(synth.make_regressor_state(sp.build_adjacency("coco", "uniform", 2, 1), seed=0), strict=True)
    tr = tr.cuda()
    _, m = _mesh_model(10475)
    aa, betas, t = _inputs(120, 55, 12, "shared", True)
    kp = SU.keypoints(torch.from_numpy(aa).cuda(), m, betas, torch.from_numpy(t).cuda())
    half = tr.hparams.win_size // 2
    dev = tr.regressor.forward_windows(kp, 2 * half + 1, offset=-half, stride=1, root=COCO_ROOT_PAIR)["poses"][:, 0]
    host = inference.run_inference(tr, kp.cpu().numpy())
    assert np.array_equal(dev.cpu().numpy(), host)
