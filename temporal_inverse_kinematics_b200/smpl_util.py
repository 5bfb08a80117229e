"""Body-model forward kinematics and mesh skinning behind the reference's ``run_smpl_inference`` signature.

Mirrors reference common/smpl_util.py:8-82.  The reference delegates to the third-party ``smplx`` package and the
licensed SMPL-X model files.  ``load_smplx_models`` reads ``SMPLX_{MALE,FEMALE,NEUTRAL}.npz`` when the directory holds
them (``SmplxBodyModel``: joints and vertices, ``return_mesh=True``) and otherwise builds *synthetic* body models
(seeded kinematic tree + rest joints + linear joint shape directions; joints only).  Joints come from the FK kernels in
libtik.so, vertices from its linear-blend-skinning kernels (``lbs``).
"""
import ctypes as C
import os

import numpy as np
import torch

from . import _lib as L

# SMPL-X body joints 0..21 (names: reference bld/syn_motion_videos.py:48-69)
SMPLX_BODY_PARENTS = [-1, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19]
SMPLX_BODY_JOINT_NAMES = ["pelvis", "left_hip", "right_hip", "spine1", "left_knee", "right_knee", "spine2",
                          "left_ankle", "right_ankle", "spine3", "left_foot", "right_foot", "neck", "left_collar",
                          "right_collar", "head", "left_shoulder", "right_shoulder", "left_elbow", "right_elbow",
                          "left_wrist", "right_wrist"]


# Full SMPL-X skeleton: 22 body joints, jaw, eyes, 2 x 15 finger joints (smplx.joint_names.JOINT_NAMES[:55];
# kinematic tree of the published SMPL-X model), followed by the five face landmarks COCO needs.  In smplx those
# landmarks are mesh vertices; without the licensed mesh they are rigid offsets from the head joint, i.e. extra leaf
# joints with identity rotation (SURVEY.md 8f row 3: "face landmarks as rigid offsets from head joint when no mesh").
_HAND = ["index1", "index2", "index3", "middle1", "middle2", "middle3", "pinky1", "pinky2", "pinky3",
         "ring1", "ring2", "ring3", "thumb1", "thumb2", "thumb3"]
SMPLX_FULL_JOINT_NAMES = (SMPLX_BODY_JOINT_NAMES + ["jaw", "left_eye_smplhf", "right_eye_smplhf"]
                          + ["left_" + h for h in _HAND] + ["right_" + h for h in _HAND])
SMPLX_FULL_PARENTS = (SMPLX_BODY_PARENTS + [15, 15, 15]
                      + [20, 25, 26, 20, 28, 29, 20, 31, 32, 20, 34, 35, 20, 37, 38]
                      + [21, 40, 41, 21, 43, 44, 21, 46, 47, 21, 49, 50, 21, 52, 53])
SMPLX_LANDMARK_NAMES = ["nose", "right_eye", "left_eye", "right_ear", "left_ear"]      # smplx JOINT_NAMES[55:60]
SMPLX_LANDMARK_PARENT = 15                                                              # head
# smplx vertex_ids["smplx"] of those landmarks (nose, reye, leye, rear, lear): what VertexJointSelector appends after joint 54
SMPLX_LANDMARK_VERTEX_IDS = [9120, 9929, 9448, 616, 6]
SMPLX_NUM_JOINTS = 55
SMPLX_NUM_BETAS = 10                                                                    # smplx.create default; the reference passes betas[:10]


def fk_body(pose, rest_joints, parents, transl=None, want_local=False, want_global=False):
    """pose (F,J,3) axis-angle or (F,J,3,3) rotation matrices, CUDA fp32; rest_joints (J,3) host array.
    Returns joints (F,J,3) [, local R (F,J,3,3)] [, global R (F,J,3,3)]."""
    if not (torch.is_tensor(pose) and pose.is_cuda):
        raise RuntimeError("fk_body: pose must be a CUDA tensor -- there is no CPU fallback")
    is_rot = pose.dim() == 4
    pose = pose.detach().float().contiguous()
    if pose.data_ptr() % 16:
        pose = pose.clone()
    F, J = pose.shape[0], pose.shape[1]
    if J > L.MAX_JOINTS:
        raise ValueError(f"fk_body supports at most {L.MAX_JOINTS} joints, got {J}")
    rest = np.ascontiguousarray(np.asarray(rest_joints, dtype=np.float32).reshape(J, 3))
    par = np.ascontiguousarray(np.asarray(parents, dtype=np.int32).reshape(J))
    joints = torch.empty((F, J, 3), dtype=torch.float32, device=pose.device)
    loc = torch.empty((F, J, 3, 3), dtype=torch.float32, device=pose.device) if want_local else None
    glo = torch.empty((F, J, 3, 3), dtype=torch.float32, device=pose.device) if want_global else None
    if transl is not None:
        transl = transl.detach().float().contiguous()
    with L.on_device(pose):
        L.check(L.lib().tik_fk_body(L.ptr(pose), int(is_rot), rest.ctypes.data_as(C.POINTER(C.c_float)),
                                    par.ctypes.data_as(C.POINTER(C.c_int32)), J, L.ptr(transl), L.ptr(joints), L.ptr(loc),
                                    L.ptr(glo), F, L.stream_ptr(pose.device)))
    out = (joints,) + ((loc,) if want_local else ()) + ((glo,) if want_global else ())
    return out[0] if len(out) == 1 else out


class SyntheticBodyModel:
    """Stand-in for an ``smplx`` body model: SMPL-X kinematic tree, seeded rest joints, and joint shape directions so
    that ``betas`` move the rest skeleton linearly (as J_regressor . shapedirs does in SMPL).

    skeleton='body' is the 22-joint tree on the IK path; skeleton='full' is the 55-joint tree plus the five face
    landmarks as rigid children of the head (60 joints), what ``smplx`` returns in ``body.joints[:, :60]``."""

    def __init__(self, gender="neutral", batch_size=1, device="cuda", seed=7, num_betas=10, skeleton="body"):
        rs = np.random.RandomState(seed + {"male": 0, "female": 1, "neutral": 2}[gender])
        self.gender, self.batch_size, self.device = gender, batch_size, device
        if skeleton == "body":
            self.parents, self.joint_names = list(SMPLX_BODY_PARENTS), list(SMPLX_BODY_JOINT_NAMES)
        elif skeleton == "full":
            self.parents = list(SMPLX_FULL_PARENTS) + [SMPLX_LANDMARK_PARENT] * len(SMPLX_LANDMARK_NAMES)
            self.joint_names = list(SMPLX_FULL_JOINT_NAMES) + list(SMPLX_LANDMARK_NAMES)
        else:
            raise ValueError("skeleton must be 'body' or 'full'")
        self.skeleton = skeleton
        J = len(self.parents)
        rest = np.zeros((J, 3))
        for i, p in enumerate(self.parents):
            off = rs.standard_normal(3) * 0.1
            rest[i] = off if p < 0 else rest[p] + off
        self.rest_joints = rest.astype(np.float32)
        self.joint_shapedirs = (rs.standard_normal((J, 3, num_betas)) * 0.01).astype(np.float32)
        self.faces = None

    def to(self, device):
        self.device = device
        return self

    def rest(self, betas=None):
        if betas is None:
            return self.rest_joints
        return self.rest_joints + self.joint_shapedirs @ np.asarray(betas, dtype=np.float32)[: self.joint_shapedirs.shape[2]]


def read_smplx_npz(path):
    """Model arrays of one SMPL-X ``.npz`` file.  Opened without pickle support and only these keys are read: real files
    also carry object arrays, which are never loaded.  Shapes and the kinematic tree are checked (``ValueError``)."""
    keys = ("v_template", "shapedirs", "posedirs", "J_regressor", "weights", "kintree_table", "f")
    with np.load(path, allow_pickle=False) as z:
        missing = [k for k in keys if k not in z.files]
        if missing:
            raise ValueError(f"{path}: missing {missing}")
        a = {k: np.asarray(z[k]) for k in keys}
    V, J = a["v_template"].shape[0], SMPLX_NUM_JOINTS
    want = {"v_template": (V, 3), "posedirs": (V, 3, (J - 1) * 9), "J_regressor": (J, V), "weights": (V, J),
            "kintree_table": (2, J)}
    for k, shp in want.items():
        if a[k].shape != shp:
            raise ValueError(f"{path}: {k} has shape {a[k].shape}, expected {shp}")
    if a["shapedirs"].ndim != 3 or a["shapedirs"].shape[:2] != (V, 3) or a["shapedirs"].shape[2] < SMPLX_NUM_BETAS:
        raise ValueError(f"{path}: shapedirs has shape {a['shapedirs'].shape}, expected ({V}, 3, >={SMPLX_NUM_BETAS})")
    if a["f"].ndim != 2 or a["f"].shape[1] != 3:
        raise ValueError(f"{path}: f has shape {a['f'].shape}, expected (n, 3)")
    if V < 1 or not np.array_equal(a["kintree_table"][0, 1:].astype(np.int64), SMPLX_FULL_PARENTS[1:J]):
        raise ValueError(f"{path}: kintree_table is not the SMPL-X tree")      # the root's entry is ignored, as smplx does
    return a


class SmplxBodyModel:
    """A body model read from an SMPL-X model file: the same surface as ``SyntheticBodyModel`` (``parents``,
    ``joint_names``, ``skeleton``, ``rest(betas)``, ``faces``) plus the mesh, skinned on the GPU by ``lbs``.

    skeleton='body': joints 0..21; skeleton='full': the 55 joints followed by the five face landmarks, which are the
    posed mesh vertices ``landmark_vertex_ids`` (smplx's VertexJointSelector; checked against V for 'full' only)."""

    def __init__(self, arrays, gender="neutral", batch_size=1, device="cuda", skeleton="body",
                 landmark_vertex_ids=SMPLX_LANDMARK_VERTEX_IDS):
        self.gender, self.batch_size, self.device = gender, batch_size, device
        if skeleton == "body":
            self.parents, self.joint_names = list(SMPLX_BODY_PARENTS), list(SMPLX_BODY_JOINT_NAMES)
        elif skeleton == "full":
            self.parents = list(SMPLX_FULL_PARENTS) + [SMPLX_LANDMARK_PARENT] * len(SMPLX_LANDMARK_NAMES)
            self.joint_names = list(SMPLX_FULL_JOINT_NAMES) + list(SMPLX_LANDMARK_NAMES)
        else:
            raise ValueError("skeleton must be 'body' or 'full'")
        self.skeleton = skeleton
        self.v_template = np.asarray(arrays["v_template"], dtype=np.float64)
        self.V = self.v_template.shape[0]
        self.landmark_vertex_ids = [int(i) for i in landmark_vertex_ids]
        if len(self.landmark_vertex_ids) != len(SMPLX_LANDMARK_NAMES) or (
                skeleton == "full" and not all(0 <= i < self.V for i in self.landmark_vertex_ids)):
            raise ValueError(f"landmark_vertex_ids must be {len(SMPLX_LANDMARK_NAMES)} vertex indices below V={self.V}")
        self.shapedirs = np.asarray(arrays["shapedirs"], dtype=np.float64)[:, :, :SMPLX_NUM_BETAS]
        self.posedirs = np.asarray(arrays["posedirs"], dtype=np.float32)
        self.J_regressor = np.asarray(arrays["J_regressor"], dtype=np.float64)
        self.weights = np.asarray(arrays["weights"], dtype=np.float32)
        self.faces = np.asarray(arrays["f"])
        # sparse skinning table: every non-zero weight of a row (exact zeros dropped, no threshold, no renormalisation)
        nz = self.weights != 0
        self.kmax = max(1, int(nz.sum(axis=1).max()))
        self.skin_idx = np.zeros((self.V, self.kmax), dtype=np.int32)
        self.skin_w = np.zeros((self.V, self.kmax), dtype=np.float32)
        for v in range(self.V):
            j = np.flatnonzero(nz[v])
            self.skin_idx[v, :len(j)] = j
            self.skin_w[v, :len(j)] = self.weights[v, j]
        self._packed, self._shaped = {}, {}

    def to(self, device):
        self.device = device
        return self

    def shaped(self, betas=None):
        """-> (v_shaped (V,3), rest joints (55,3)), float64: v_template + shapedirs[..., :10] . betas and its J_regressor."""
        v = self.v_template
        if betas is not None:
            b = np.asarray(betas, dtype=np.float64).reshape(-1)
            if b.shape[0] > SMPLX_NUM_BETAS:
                raise ValueError(f"at most {SMPLX_NUM_BETAS} betas, got {b.shape[0]}")
            v = v + self.shapedirs[:, :, :b.shape[0]] @ b
        return v, self.J_regressor @ v

    def rest(self, betas=None):
        """Rest joints (55,3) fp32 for ``betas`` (None: the template)."""
        return self.shaped(betas)[1].astype(np.float32)

    def device_shape(self, betas, device):
        """(v_shaped, rest joints) as CUDA fp32 tensors plus the rest joints on the host, cached per betas."""
        key = (str(device), None if betas is None else np.asarray(betas, dtype=np.float32).reshape(-1).tobytes())
        if key not in self._shaped:
            if len(self._shaped) >= 16:
                self._shaped.clear()
            v, j = self.shaped(betas)
            j32 = np.ascontiguousarray(j, dtype=np.float32)
            self._shaped[key] = (torch.from_numpy(v.astype(np.float32)).to(device), torch.from_numpy(j32).to(device), j32)
        return self._shaped[key]

    def device_pack(self, dtype, device):
        """posedirs as the (ceil(3V/128)*128, 512) K-contiguous operand in ``dtype`` and the sparse skinning table, on
        ``device``; packed once per (dtype, device)."""
        key = (dtype, str(device))
        if key not in self._packed:
            rows = -(-3 * self.V // 128) * 128
            pd = np.zeros((rows, 512), dtype=np.float32)
            pd[:3 * self.V, :self.posedirs.shape[2]] = self.posedirs.reshape(3 * self.V, -1)
            t = torch.from_numpy(pd).to(device)
            self._packed[key] = (t.to(torch.bfloat16) if dtype == "bf16" else t, torch.from_numpy(self.skin_idx).to(device),
                                 torch.from_numpy(self.skin_w).to(device))
        return self._packed[key]


def load_smplx_models(smplx_dir, device, batch_size, skeleton="body"):
    """Same signature as reference common/smpl_util.py:8-19.  With ``smplx_dir`` holding SMPLX_{MALE,FEMALE,NEUTRAL}.npz
    (the reference's file names) the models are read from them (``SmplxBodyModel``, joints and vertices); with None or a
    directory without them, synthetic models (joints only).  skeleton='full' gives the 55 joints + five face landmarks
    (SURVEY.md 8f row 3)."""
    genders = ("male", "female", "neutral")
    if smplx_dir is not None:
        paths = {g: os.path.join(smplx_dir, f"SMPLX_{g.upper()}.npz") for g in genders}
        present = [g for g in genders if os.path.exists(paths[g])]
        if present and len(present) < len(genders):
            raise FileNotFoundError(f"{smplx_dir} holds only {[os.path.basename(paths[g]) for g in present]}")
        if present:
            return {g: SmplxBodyModel(read_smplx_npz(paths[g]), g, batch_size, device, skeleton=skeleton) for g in genders}
    return {g: SyntheticBodyModel(g, batch_size, device, skeleton=skeleton) for g in genders}


def lbs(pose, model, betas=None, transl=None, dtype="fp32"):
    """SMPL-X forward of a ``SmplxBodyModel`` on the GPU (smplx.lbs.lbs + VertexJointSelector + transl).
    pose (F, 22 | 55 | 60, 3) axis-angle CUDA tensor (22: body only, hands / jaw / eyes identity; 60: joints past 54
    ignored); betas up to 10 values or None; transl (F,3) CUDA tensor or None; dtype 'fp32' (3xTF32 pose blend, 1e-4
    parity) or 'bf16' (bf16 pose-blend operands).  Returns joints (F, len(model.parents), 3) and vertices (F, V, 3), fp32
    CUDA tensors."""
    if not (torch.is_tensor(pose) and pose.is_cuda):
        raise RuntimeError("lbs: pose must be a CUDA tensor -- there is no CPU fallback")
    if transl is not None and not (torch.is_tensor(transl) and transl.is_cuda):
        raise RuntimeError("lbs: transl must be a CUDA tensor -- there is no CPU fallback")
    if not isinstance(model, SmplxBodyModel):
        raise TypeError("lbs needs a SmplxBodyModel (a model read from an SMPL-X file)")
    if pose.dim() != 3 or pose.shape[1] not in (22, SMPLX_NUM_JOINTS, 60) or pose.shape[2] != 3:
        raise ValueError(f"lbs: pose must be (F, 22 | 55 | 60, 3), got {tuple(pose.shape)}")
    F = pose.shape[0]
    if transl is not None and tuple(transl.shape) != (F, 3):
        raise ValueError(f"lbs: transl must be ({F}, 3), got {tuple(transl.shape)}")
    if dtype not in ("fp32", "bf16"):
        raise ValueError(f"lbs: dtype must be 'fp32' or 'bf16', got {dtype!r}")
    dev = pose.device
    pose = pose.detach().float()
    if pose.shape[1] == 22:                                      # full_pose_from_amass of a 66-column pose
        pose = torch.cat([pose, pose.new_zeros(F, SMPLX_NUM_JOINTS - 22, 3)], dim=1)
    pose = pose[:, :SMPLX_NUM_JOINTS].contiguous()
    if transl is not None:
        transl = transl.detach().float().contiguous()
    v_shaped, rest_dev, rest_host = model.device_shape(betas, dev)
    posedirs, skin_idx, skin_w = model.device_pack(dtype, dev)
    Jo = len(model.parents)
    joints = torch.empty((F, Jo, 3), dtype=torch.float32, device=dev)
    verts = torch.empty((F, model.V, 3), dtype=torch.float32, device=dev)
    if F == 0:
        return joints, verts
    fk_j, fk_loc, fk_glo = fk_body(pose, rest_host, SMPLX_FULL_PARENTS[:SMPLX_NUM_JOINTS], want_local=True, want_global=True)
    m = L.TikLbsModel()
    m.V, m.J, m.kmax = model.V, SMPLX_NUM_JOINTS, model.kmax
    if model.skeleton == "full":
        m.n_landmarks = len(model.landmark_vertex_ids)
        for k, v in enumerate(model.landmark_vertex_ids):
            m.landmark_vid[k] = v
    m.v_shaped_dev, m.rest_joints_dev, m.posedirs_dev = v_shaped.data_ptr(), rest_dev.data_ptr(), posedirs.data_ptr()
    m.skin_idx_dev, m.skin_w_dev = skin_idx.data_ptr(), skin_w.data_ptr()
    dt = L.TIK_BF16 if dtype == "bf16" else L.TIK_F32
    nbytes = L.i64()
    with L.on_device(pose):
        L.check(L.lib().tik_lbs_workspace_bytes(C.byref(m), dt, F, C.byref(nbytes)))
        ws = torch.empty(max(1, nbytes.value), dtype=torch.uint8, device=dev)
        L.check(L.lib().tik_lbs(C.byref(m), dt, L.ptr(fk_j), L.ptr(fk_loc), L.ptr(fk_glo), SMPLX_NUM_JOINTS, L.ptr(transl), F,
                                L.ptr(ws), nbytes.value, L.ptr(verts), L.ptr(joints), Jo, L.stream_ptr(dev)))
    return joints, verts


def full_pose_from_amass(poses, n_joints):
    """AMASS / reference pose rows (F, 66 | 156 | 165): root + body [0:66], left hand [66:111], right hand [111:156]
    (common/smpl_util.py:61-64) -> (F, n_joints, 3) in SMPL-X joint order; jaw, eyes and landmark pseudo-joints get a
    zero (identity) rotation exactly as ``smplx`` defaults them."""
    poses = np.asarray(poses, dtype=np.float32)
    F = poses.shape[0]
    out = np.zeros((F, n_joints, 3), dtype=np.float32)
    out[:, :22] = poses[:, :66].reshape(F, 22, 3)
    if n_joints >= 55 and poses.shape[1] >= 156:
        out[:, 25:40] = poses[:, 66:111].reshape(F, 15, 3)
        out[:, 40:55] = poses[:, 111:156].reshape(F, 15, 3)
    return out


def run_smpl_inference(data, smplx_models, device, apply_trans=True, apply_root_rot=True, apply_shape=True,
                       return_mesh=False):
    """data: {'poses': (F, >=66) axis-angle, 'gender', ['trans' (F,3)], ['betas']} -> joints (F, J, 3) numpy
    (J = 22 for body models, 60 for skeleton='full' models: 55 SMPL-X joints + 5 face landmarks), or (joints, vertices
    (F, V, 3)) with return_mesh=True, which needs a model read from an SMPL-X file (``SmplxBodyModel``).
    Reference common/smpl_util.py:22-82; the fixed-batch padding loop there is unnecessary here (one launch)."""
    model = smplx_models[str(data["gender"])]
    mesh = isinstance(model, SmplxBodyModel)
    if return_mesh and not mesh:
        raise NotImplementedError("vertices need an SMPL-X model file: load_smplx_models(dir) with SMPLX_*.npz in dir")
    J = len(model.parents)
    if J == 22 and not return_mesh:
        poses = torch.as_tensor(np.asarray(data["poses"], dtype=np.float32)[:, :66]).to(device).view(-1, 22, 3).contiguous()
    else:                                                         # full skeleton / mesh: body + hands (+ identity jaw / eyes / landmarks)
        poses = torch.as_tensor(full_pose_from_amass(data["poses"], SMPLX_NUM_JOINTS if mesh else J)).to(device)
    if not apply_root_rot:
        poses = poses.clone()
        poses[:, 0] = 0
    transl = torch.as_tensor(np.asarray(data["trans"], dtype=np.float32)).to(device) if apply_trans else None
    betas = np.asarray(data["betas"])[:10] if apply_shape else None
    if mesh and (return_mesh or J != 22):                         # landmark joints are mesh vertices
        joints, verts = lbs(poses, model, betas, transl)
        return (joints.cpu().numpy(), verts.cpu().numpy()) if return_mesh else joints.cpu().numpy()
    rest = model.rest(betas)[:J]
    return fk_body(poses, rest, model.parents, transl).cpu().numpy()


def smplx_joints_to_coco(joints, joint_names):
    """(F, J, 3) joints of the full skeleton -> (F, 17, 3) COCO keypoints, the gather of
    common/keypoints_util.py:27-60 applied to FK output (SURVEY.md 8f row 3)."""
    from .keypoints_util import convert_seq_keypoints, generate_smplx_to_coco_mappings
    return convert_seq_keypoints(joints, generate_smplx_to_coco_mappings(list(joint_names)))
