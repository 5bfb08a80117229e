"""SMPL-X mesh skinning (run_smpl_inference(return_mesh=True), smpl_util.lbs, tik_lbs): the fp64 oracle's properties and
its agreement with an independent homogeneous formulation, the model-file loader, the device packing, and on the GPU the
kernels against the oracle, the inference entry point, guard regions and CUDA-graph replay.  Parity with smplx itself is
unpinned (third-party package, licensed model files), as for FK: the model files here are synthetic (oracle/smplx_synth.py)."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import lbs_port, lbs_scipy, smplx_synth
from oracle.geometry_port import batch_rodrigues
from temporal_inverse_kinematics_b200 import smpl_util as SU

PARENTS55 = smplx_synth.PARENTS55
TOL = 1e-4
# bf16 pose-blend operands at V = 10,475 (measured on the B200, DESIGN.md section 4): max-abs and RMS over all vertex
# coordinates against the fp64 oracle
BF16_MAX, BF16_RMS = 2e-3, 3e-4


def _model_dict(arrays):
    return dict(arrays, parents=PARENTS55)


def _pose(F, seed, scale=0.4):
    return np.random.RandomState(seed).standard_normal((F, 55, 3)) * scale


# ------------------------------------------------------------------ oracle


def test_oracle_zero_pose_zero_posedirs_gives_v_shaped():
    a = smplx_synth.make_smplx_arrays(60, seed=1)
    a["posedirs"] = np.zeros_like(a["posedirs"])
    betas = np.linspace(-1, 1, 10)
    _, verts = lbs_port.lbs(np.zeros((2, 55, 3)), _model_dict(a), betas)
    v_shaped, _ = lbs_port.shape(a["v_template"], a["shapedirs"], a["J_regressor"], betas)
    assert np.abs(verts - v_shaped).max() < 1e-12


def test_oracle_root_rotation_is_rigid_about_the_root():
    a = smplx_synth.make_smplx_arrays(60, seed=2)
    aa = np.zeros((3, 55, 3))
    aa[:, 0] = np.random.RandomState(0).standard_normal((3, 3))
    joints, verts = lbs_port.lbs(aa, _model_dict(a))
    v, J = lbs_port.shape(a["v_template"], a["shapedirs"], a["J_regressor"])
    R = batch_rodrigues(aa[:, 0]).reshape(-1, 3, 3)
    want = np.einsum("fab,vb->fva", R, v - J[0]) + J[0]
    assert np.abs(verts - want).max() < 1e-12
    assert np.abs(joints - (np.einsum("fab,jb->fja", R, J - J[0]) + J[0])).max() < 1e-12


def test_oracle_one_hot_vertex_follows_its_joint():
    a = smplx_synth.make_smplx_arrays(60, seed=3)
    a["posedirs"] = np.zeros_like(a["posedirs"])
    for v, j in ((0, 0), (1, 20), (2, 54), (3, 15)):
        a["weights"][v] = 0
        a["weights"][v, j] = 1
    aa = _pose(4, 5)
    joints, verts = lbs_port.lbs(aa, _model_dict(a))
    v_shaped, J = lbs_port.shape(a["v_template"], a["shapedirs"], a["J_regressor"])
    R = batch_rodrigues(aa.reshape(-1, 3)).reshape(4, 55, 3, 3)
    from oracle.fk_port import forward_kinematics
    _, gR = forward_kinematics(R, J, PARENTS55)
    for v, j in ((0, 0), (1, 20), (2, 54), (3, 15)):
        want = np.einsum("fab,b->fa", gR[:, j], v_shaped[v] - J[j]) + joints[:, j]
        assert np.abs(verts[:, v] - want).max() < 1e-12


def test_oracle_pose_offsets_are_linear_in_posedirs():
    a = smplx_synth.make_smplx_arrays(40, seed=4)
    rs = np.random.RandomState(1)
    P1, P2 = rs.standard_normal(a["posedirs"].shape), rs.standard_normal(a["posedirs"].shape)
    feat = lbs_port.pose_feature(batch_rodrigues(_pose(3, 6).reshape(-1, 3)).reshape(3, 55, 3, 3))
    lhs = lbs_port.pose_offsets(feat, 2.0 * P1 - 0.5 * P2)
    rhs = 2.0 * lbs_port.pose_offsets(feat, P1) - 0.5 * lbs_port.pose_offsets(feat, P2)
    assert np.abs(lhs - rhs).max() < 1e-12
    zero_feat = lbs_port.pose_feature(np.broadcast_to(np.eye(3), (1, 55, 3, 3)))
    assert not zero_feat.any()
    # and the synthetic posedirs matter at test poses: offsets of several centimetres
    assert np.abs(lbs_port.pose_offsets(feat, a["posedirs"])).max() > 0.03


def test_oracle_transl_shifts_everything():
    a = _model_dict(smplx_synth.make_smplx_arrays(30, seed=5))
    aa, tr = _pose(3, 7), np.random.RandomState(2).standard_normal((3, 3))
    j0, v0 = lbs_port.lbs(aa, a)
    j1, v1 = lbs_port.lbs(aa, a, transl=tr)
    assert np.abs(j1 - j0 - tr[:, None]).max() < 1e-12 and np.abs(v1 - v0 - tr[:, None]).max() < 1e-12


def test_oracle_matches_homogeneous_formulation():
    a = _model_dict(smplx_synth.make_smplx_arrays(200, seed=6))
    aa, tr, betas = _pose(5, 8, 0.6), np.random.RandomState(3).standard_normal((5, 3)), np.linspace(-2, 2, 10)
    j0, v0 = lbs_port.lbs(aa, a, betas, tr)
    j1, v1 = lbs_scipy.lbs_homogeneous(batch_rodrigues(aa.reshape(-1, 3)).reshape(5, 55, 3, 3), a, betas, tr)
    assert np.abs(j0 - j1).max() < 1e-9 and np.abs(v0 - v1).max() < 1e-9


# ------------------------------------------------------------------ loader and packing


def test_loader_round_trips_a_written_file(tmp_path):
    arrays = smplx_synth.write_smplx_dir(str(tmp_path), 50, seed=10)
    models = SU.load_smplx_models(str(tmp_path), "cuda", 4)
    assert set(models) == {"male", "female", "neutral"}
    for g, m in models.items():
        a = arrays[g]
        assert isinstance(m, SU.SmplxBodyModel) and m.gender == g and m.V == 50 and m.skeleton == "body"
        assert np.array_equal(m.faces, a["f"]) and np.array_equal(m.v_template, a["v_template"])
        assert len(m.parents) == len(m.joint_names) == 22
        betas = np.linspace(-1, 1, 10)
        _, want = lbs_port.shape(a["v_template"], a["shapedirs"], a["J_regressor"], betas)
        assert np.abs(m.rest(betas) - want).max() < 1e-6
    with pytest.raises(ValueError, match="landmark"):              # V = 50 holds no smplx landmark vertices
        SU.load_smplx_models(str(tmp_path), "cuda", 4, skeleton="full")
    assert all(isinstance(m, SU.SyntheticBodyModel) for m in SU.load_smplx_models(None, "cuda", 4).values())
    assert all(isinstance(m, SU.SyntheticBodyModel) for m in SU.load_smplx_models(str(tmp_path / "nothing"), "cuda", 4).values())
    (tmp_path / "SMPLX_MALE.npz").unlink()
    with pytest.raises(FileNotFoundError):
        SU.load_smplx_models(str(tmp_path), "cuda", 4)


def test_loader_never_loads_object_arrays(tmp_path):
    p = str(tmp_path / "m.npz")
    smplx_synth.write_smplx_npz(p, 20, seed=11, with_object_key=True)
    with np.load(p, allow_pickle=False) as z:
        assert "part2num" in z.files
        with pytest.raises(ValueError):
            z["part2num"]                                         # noqa: B018  the key is really pickled
    a = SU.read_smplx_npz(p)
    assert "part2num" not in a and a["v_template"].shape == (20, 3)


@pytest.mark.parametrize("key,bad", [
    ("kintree_table", lambda a: np.stack([np.r_[a["kintree_table"][0, :5], 0, a["kintree_table"][0, 6:]], a["kintree_table"][1]])),
    ("posedirs", lambda a: a["posedirs"][:, :, :480]),
    ("shapedirs", lambda a: a["shapedirs"][:, :, :9]),
    ("J_regressor", lambda a: a["J_regressor"][:54]),
    ("weights", lambda a: a["weights"][:-1]),
    ("f", lambda a: a["f"][:, :2]),
    ("v_template", lambda a: a["v_template"][:, :2]),
])
def test_loader_rejects_bad_files(tmp_path, key, bad):
    a = smplx_synth.make_smplx_arrays(20, seed=12)
    a[key] = bad(a)
    p = str(tmp_path / "bad.npz")
    np.savez(p, **a)
    with pytest.raises(ValueError):
        SU.read_smplx_npz(p)
    del a[key]
    np.savez(p, **a)
    with pytest.raises(ValueError, match="missing"):
        SU.read_smplx_npz(p)


def test_packing_matches_oracle_order():
    a = smplx_synth.make_smplx_arrays(45, seed=13)
    m = SU.SmplxBodyModel(a, skeleton="body", landmark_vertex_ids=[0, 1, 2, 3, 4])
    pd, idx, w = m.device_pack("fp32", "cpu")
    assert pd.shape == (256, 512) and not pd[135:].any() and not pd[:, 486:].any()
    R = batch_rodrigues(_pose(3, 9).reshape(-1, 3)).reshape(3, 55, 3, 3)
    feat = lbs_port.pose_feature(R)
    got = (feat @ pd.double().numpy()[:135, :486].T).reshape(3, 45, 3)
    assert np.abs(got - lbs_port.pose_offsets(feat, a["posedirs"].astype(np.float32))).max() < 1e-12
    # the kernel's feature column 9 (j - 1) + 3 a + b is R_j[a, b] - I[a, b]
    assert feat[0, 9 * 4 + 3 * 1 + 2] == R[0, 5, 1, 2] and feat[0, 9 * 0 + 4] == R[0, 1, 1, 1] - 1
    dense = np.zeros((45, 55), np.float32)
    for v in range(45):
        for k in range(m.kmax):
            dense[v, idx[v, k]] += w[v, k].item()
    assert np.array_equal(dense, a["weights"].astype(np.float32))
    assert m.kmax == int((a["weights"] != 0).sum(1).max()) and 1 <= m.kmax <= 4
    assert m.device_pack("bf16", "cpu")[0].dtype == torch.bfloat16
    with pytest.raises(ValueError):
        SU.SmplxBodyModel(a, skeleton="full", landmark_vertex_ids=[0, 1, 2, 3, 45])      # out of range for V = 45


def test_lbs_has_no_cpu_fallback():
    m = SU.SmplxBodyModel(smplx_synth.make_smplx_arrays(10, seed=14), landmark_vertex_ids=[0, 1, 2, 3, 4])
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        SU.lbs(torch.zeros(2, 55, 3), m)


# ------------------------------------------------------------------ GPU


_MODELS = {}


def _mesh_model(V, skeleton="body"):
    if (V, skeleton) not in _MODELS:
        a = smplx_synth.make_smplx_arrays(V, seed=V)
        lm = SU.SMPLX_LANDMARK_VERTEX_IDS if V > max(SU.SMPLX_LANDMARK_VERTEX_IDS) else [v % V for v in (3, 1, 4, 1, 5)]
        _MODELS[(V, skeleton)] = (a, SU.SmplxBodyModel(a, skeleton=skeleton, landmark_vertex_ids=lm))
    return _MODELS[(V, skeleton)]


def _inputs(F, seed, with_betas, with_transl):
    rs = np.random.RandomState(seed)
    aa = rs.standard_normal((F, 55, 3)).astype(np.float32) * 0.4
    betas = rs.standard_normal(10).astype(np.float32) if with_betas else None
    tr = rs.standard_normal((F, 3)).astype(np.float32) if with_transl else None
    return aa, betas, tr


# chunks: V = 10,475 runs 256 frames per chunk, V <= 37 1024 (805 = 3 chunks + 37, 2500 = 2 chunks + 452)
@pytest.mark.gpu
@pytest.mark.parametrize("V,F,with_betas,with_transl", [
    (1, 1, False, False), (1, 7, True, True), (37, 1, True, False), (37, 7, False, True), (37, 255, True, True),
    (37, 257, False, False), (37, 2500, True, True), (10475, 1, True, True), (10475, 7, False, False),
    (10475, 255, False, True), (10475, 257, True, False), (10475, 805, True, True),
])
def test_lbs_fp32_matches_oracle(V, F, with_betas, with_transl):
    a, m = _mesh_model(V, "full")
    aa, betas, tr = _inputs(F, V + F, with_betas, with_transl)
    joints, verts = SU.lbs(torch.from_numpy(aa).cuda(), m, betas, None if tr is None else torch.from_numpy(tr).cuda())
    ej, ev = lbs_port.lbs(aa, _model_dict(a), betas, tr)
    assert joints.shape == (F, 60, 3) and verts.shape == (F, V, 3)
    assert np.abs(verts.cpu().numpy() - ev).max() < TOL
    j = joints.cpu().numpy()
    assert np.abs(j[:, :55] - ej).max() < TOL
    assert np.abs(j[:, 55:] - ev[:, m.landmark_vertex_ids]).max() < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("F", [257, 1100])
def test_lbs_bf16_tolerance(F):
    a, m = _mesh_model(10475)
    aa, betas, tr = _inputs(F, 77 + F, True, True)
    joints, verts = SU.lbs(torch.from_numpy(aa).cuda(), m, betas, torch.from_numpy(tr).cuda(), dtype="bf16")
    ej, ev = lbs_port.lbs(aa, _model_dict(a), betas, tr)
    d = verts.cpu().numpy() - ev
    err_max, err_rms = float(np.abs(d).max()), float(np.sqrt((d ** 2).mean()))
    print(f"bf16 V=10475 F={F}: max-abs {err_max:.3e} m, RMS {err_rms:.3e} m")
    assert err_max < BF16_MAX and err_rms < BF16_RMS, (err_max, err_rms)
    assert np.abs(joints.cpu().numpy() - ej[:, :22]).max() < TOL                 # joints do not go through the blend


@pytest.mark.gpu
def test_lbs_argument_errors_and_pose_widths():
    a, m = _mesh_model(37)
    with pytest.raises(ValueError):
        SU.lbs(torch.zeros(3, 54, 3, device="cuda"), m)
    with pytest.raises(ValueError):
        SU.lbs(torch.zeros(3, 55, 3, device="cuda"), m, transl=torch.zeros(2, 3, device="cuda"))
    with pytest.raises(ValueError):
        SU.lbs(torch.zeros(3, 55, 3, device="cuda"), m, dtype="fp16")
    with pytest.raises(RuntimeError):
        SU.lbs(torch.zeros(3, 55, 3, device="cuda"), m, transl=torch.zeros(3, 3))
    with pytest.raises(TypeError):
        SU.lbs(torch.zeros(3, 55, 3, device="cuda"), SU.SyntheticBodyModel())
    j0, v0 = SU.lbs(torch.zeros(0, 55, 3, device="cuda"), m)
    assert j0.shape == (0, 22, 3) and v0.shape == (0, 37, 3)
    aa = _pose(9, 3).astype(np.float32)
    aa[:, 22:] = 0
    _, v55 = SU.lbs(torch.from_numpy(aa).cuda(), m)
    _, v22 = SU.lbs(torch.from_numpy(np.ascontiguousarray(aa[:, :22])).cuda(), m)
    _, v60 = SU.lbs(torch.from_numpy(np.concatenate([aa, np.ones((9, 5, 3), np.float32)], 1)).cuda(), m)
    assert torch.equal(v55, v22) and torch.equal(v55, v60)


@pytest.mark.gpu
@pytest.mark.parametrize("skeleton", ["body", "full"])
def test_run_smpl_inference_return_mesh(tmp_path, skeleton):
    arrays = smplx_synth.write_smplx_dir(str(tmp_path), 10475, seed=20)
    models = SU.load_smplx_models(str(tmp_path), "cuda", 8, skeleton=skeleton)
    rs = np.random.RandomState(4)
    F = 40
    data = {"poses": (rs.standard_normal((F, 156)) * 0.3).astype(np.float32), "gender": "female",
            "trans": rs.standard_normal((F, 3)).astype(np.float32), "betas": rs.standard_normal(16).astype(np.float32)}
    a = _model_dict(arrays["female"])
    m = models["female"]
    aa = SU.full_pose_from_amass(data["poses"], 55)
    J = 22 if skeleton == "body" else 60
    for trans, root, shape in ((True, True, True), (False, True, False), (True, False, True), (False, False, False)):
        joints, verts = SU.run_smpl_inference(data, models, "cuda", apply_trans=trans, apply_root_rot=root, apply_shape=shape,
                                              return_mesh=True)
        p = aa.copy()
        if not root:
            p[:, 0] = 0
        ej, ev = lbs_port.lbs(p, a, data["betas"][:10] if shape else None, data["trans"] if trans else None)
        assert joints.shape == (F, J, 3) and verts.shape == (F, 10475, 3)
        assert np.abs(verts - ev).max() < TOL and np.abs(joints[:, :min(J, 55)] - ej[:, :min(J, 55)]).max() < TOL
        if skeleton == "full":
            assert np.array_equal(joints[:, 55:], verts[:, SU.SMPLX_LANDMARK_VERTEX_IDS])
        only = SU.run_smpl_inference(data, models, "cuda", apply_trans=trans, apply_root_rot=root, apply_shape=shape)
        assert np.abs(only - joints).max() < TOL
    if skeleton == "full":
        coco = SU.smplx_joints_to_coco(joints, m.joint_names)
        assert np.array_equal(coco[:, 0], verts[:, 9120]) and np.array_equal(coco[:, 1], verts[:, 9448])   # nose, left eye
        assert np.array_equal(coco[:, 3], verts[:, 6]) and np.array_equal(coco[:, 9], joints[:, 20])       # left ear, wrist


def _raw_inputs(m, F, seed, dtype):
    aa = torch.from_numpy(_pose(F, seed).astype(np.float32)).cuda()
    tr = torch.randn(F, 3, device="cuda")
    v_shaped, rest_dev, rest_host = m.device_shape(None, torch.device("cuda"))
    pd, idx, w = m.device_pack(dtype, torch.device("cuda"))
    fk = SU.fk_body(aa, rest_host, PARENTS55, want_local=True, want_global=True)
    from temporal_inverse_kinematics_b200 import _lib as L
    s = L.TikLbsModel()
    s.V, s.J, s.kmax, s.n_landmarks = m.V, 55, m.kmax, 5
    for k, v in enumerate(m.landmark_vertex_ids):
        s.landmark_vid[k] = v
    s.v_shaped_dev, s.rest_joints_dev, s.posedirs_dev = v_shaped.data_ptr(), rest_dev.data_ptr(), pd.data_ptr()
    s.skin_idx_dev, s.skin_w_dev = idx.data_ptr(), w.data_ptr()
    nb = L.i64()
    L.check(L.lib().tik_lbs_workspace_bytes(C.byref(s), L.TIK_BF16 if dtype == "bf16" else L.TIK_F32, F, C.byref(nb)))
    return L, s, fk, tr, nb.value


@pytest.mark.gpu
def test_lbs_writes_only_its_outputs():
    """Vertex and joint outputs carved out of sentinel-filled buffers, for F around the 32-frame tile and the 256-frame
    fp32 chunk at V = 10,475, and V around the 32-vertex tile."""
    GUARD, SENT = 4096, 12345.0
    for V, frames in ((10475, (31, 32, 33, 256, 257)), (31, (1, 33)), (32, (32, 1025)), (33, (65,)), (1, (3,))):
        _, m = _mesh_model(V, "full")
        for F in frames:
            L, s, (fj, fl, fg), tr, nb = _raw_inputs(m, F, V + F, "fp32")
            ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
            vb = torch.full((GUARD + F * V * 3 + GUARD,), SENT, device="cuda")
            jb = torch.full((GUARD + F * 60 * 3 + GUARD,), SENT, device="cuda")
            vo, jo = vb[GUARD:GUARD + F * V * 3], jb[GUARD:GUARD + F * 60 * 3]
            L.check(L.lib().tik_lbs(C.byref(s), L.TIK_F32, L.ptr(fj), L.ptr(fl), L.ptr(fg), 55, L.ptr(tr), F, L.ptr(ws), nb,
                                    L.ptr(vo), L.ptr(jo), 60, L.stream_ptr()))
            torch.cuda.synchronize()
            for buf, n in ((vb, F * V * 3), (jb, F * 60 * 3)):
                assert bool((buf[:GUARD] == SENT).all()) and bool((buf[GUARD + n:] == SENT).all()), (V, F)
                inner = buf[GUARD:GUARD + n]
                assert bool(torch.isfinite(inner).all()) and not bool((inner == SENT).any()), (V, F)
            assert L.lib().tik_lbs(C.byref(s), L.TIK_F32, L.ptr(fj), L.ptr(fl), L.ptr(fg), 55, L.ptr(tr), F, L.ptr(ws), nb - 256,
                                   L.ptr(vo), L.ptr(jo), 60, L.stream_ptr()) == L._H["TIK_ERR_WORKSPACE"]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_lbs_cuda_graph_replay_is_bit_exact(dtype):
    _, m = _mesh_model(10475, "full")
    F = 300
    L, s, (fj, fl, fg), tr, nb = _raw_inputs(m, F, 5, dtype)
    dt = L.TIK_BF16 if dtype == "bf16" else L.TIK_F32
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    eager_v, eager_j = torch.empty(F, m.V, 3, device="cuda"), torch.empty(F, 60, 3, device="cuda")
    graph_v, graph_j = torch.zeros_like(eager_v), torch.zeros_like(eager_j)

    def run(v, j):
        L.check(L.lib().tik_lbs(C.byref(s), dt, L.ptr(fj), L.ptr(fl), L.ptr(fg), 55, L.ptr(tr), F, L.ptr(ws), nb, L.ptr(v),
                                L.ptr(j), 60, L.stream_ptr()))
    run(eager_v, eager_j)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        run(graph_v, graph_j)
    g.replay()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(graph_v, eager_v) and torch.equal(graph_j, eager_j)
