"""Body-model forward kinematics and mesh skinning behind the reference's ``run_smpl_inference`` signature.

Mirrors reference common/smpl_util.py:8-82.  The reference delegates to the third-party ``smplx`` package and the
licensed SMPL-X model files.  ``load_smplx_models`` reads ``SMPLX_{MALE,FEMALE,NEUTRAL}.npz`` when the directory holds
them (``SmplxBodyModel``: joints and vertices, ``return_mesh=True``) and otherwise builds *synthetic* body models
(seeded kinematic tree + rest joints + linear joint shape directions; joints only).  Joints come from the FK kernels in
libtik.so, vertices from its linear-blend-skinning kernels (``lbs``), and keypoints (joints + face landmarks, e.g.
COCO-17) from one kernel that never skins the mesh (``keypoints``, ``run_smpl_keypoints``).
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

    def check_keypoints(self):
        """``ValueError`` unless the model has the face landmarks ``keypoints`` needs (skeleton='full')."""
        if self.skeleton != "full":
            raise ValueError("keypoints need skeleton='full' (the body skeleton has no face landmarks)")

    def keypoint_pack(self, device):
        """The model as ``tik_body_keypoints`` reads it, cached per device: the 55 joints' rest positions and shape
        directions, the five landmarks as points skinned with weight 1 to the head and no pose blend -- the rigid
        landmark children of the 60-joint tree.  skeleton='body' has no landmarks (``ValueError``)."""
        self.check_keypoints()
        key = str(device)
        if key not in getattr(self, "_kp", {}):
            J, L = SMPLX_NUM_JOINTS, len(SMPLX_LANDMARK_NAMES)
            self._kp = getattr(self, "_kp", {})
            self._kp[key] = KeypointPack(device, self.rest_joints[:J], self.joint_shapedirs[:J], self.rest_joints[J:],
                                         self.joint_shapedirs[J:], None, np.full((L, 1), SMPLX_LANDMARK_PARENT),
                                         np.ones((L, 1)))
        return self._kp[key]


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

    def check_keypoints(self):
        """``ValueError`` unless every landmark id is a vertex of the model (whatever the skeleton)."""
        if not all(0 <= i < self.V for i in self.landmark_vertex_ids):
            raise ValueError(f"landmark_vertex_ids {self.landmark_vertex_ids} must be vertex indices below V={self.V}")

    def keypoint_pack(self, device):
        """The model as ``tik_body_keypoints`` reads it, cached per device: Jt = J_regressor . v_template, Jd =
        J_regressor . shapedirs[..., :10] (fp64, rounded once), and the rows of ``landmark_vertex_ids``: template,
        shape directions, posedirs and skinning table.  ``ValueError`` when a landmark id is not below V."""
        self.check_keypoints()
        key = str(device)
        if key not in getattr(self, "_kp", {}):
            ids = self.landmark_vertex_ids
            nz = (self.skin_w[ids] != 0).sum(axis=1)
            kmax = max(1, int(nz.max()))
            self._kp = getattr(self, "_kp", {})
            self._kp[key] = KeypointPack(device, self.J_regressor @ self.v_template,
                                         np.einsum("jv,vck->jck", self.J_regressor, self.shapedirs), self.v_template[ids],
                                         self.shapedirs[ids], self.posedirs[ids].reshape(3 * len(ids), -1),
                                         self.skin_idx[ids, :kmax], self.skin_w[ids, :kmax])
        return self._kp[key]


class KeypointPack:
    """Device arrays of one body model for ``tik_body_keypoints`` and the ``TikKeypointModel`` that points at them
    (``.c``).  Points 0..54 are the SMPL-X joints, 55.. the landmarks."""

    def __init__(self, device, jt, jd, lm_t, lm_d, lm_posedirs, skin_idx, skin_w):
        def dev(a, dt=torch.float32):
            return torch.from_numpy(np.ascontiguousarray(a)).to(dt).to(device)
        self.n_betas = int(jd.shape[2])
        if self.n_betas > L.KP_MAX_BETAS:
            raise ValueError(f"at most {L.KP_MAX_BETAS} shape directions, got {self.n_betas}")
        self.jt, self.jd, self.lm_t, self.lm_d = dev(jt), dev(jd), dev(lm_t), dev(lm_d)
        self.lm_posedirs = None if lm_posedirs is None else dev(lm_posedirs)
        self.skin_idx, self.skin_w = dev(skin_idx, torch.int32), dev(skin_w)
        self.n_landmarks, self.kmax = int(lm_t.shape[0]), int(skin_idx.shape[1])
        c = L.TikKeypointModel()
        c.n_betas, c.n_landmarks, c.kmax = self.n_betas, self.n_landmarks, self.kmax
        c.joint_template_dev, c.joint_dirs_dev = self.jt.data_ptr(), self.jd.data_ptr() if self.n_betas else None
        c.lm_template_dev, c.lm_dirs_dev = self.lm_t.data_ptr(), self.lm_d.data_ptr() if self.n_betas else None
        c.lm_posedirs_dev = None if self.lm_posedirs is None else self.lm_posedirs.data_ptr()
        c.lm_skin_idx_dev, c.lm_skin_w_dev = self.skin_idx.data_ptr(), self.skin_w.data_ptr()
        self.c = c


def keypoint_names():
    """Names of the points ``keypoints`` can select: the 55 SMPL-X joints, then the five face landmarks."""
    return list(SMPLX_FULL_JOINT_NAMES) + list(SMPLX_LANDMARK_NAMES)


def keypoint_indices(select="coco"):
    """'coco' (the order of generate_smplx_to_coco_mappings over the 60 full-skeleton names) or a list of point names
    -> point indices.  ``ValueError`` for an unknown name or a selection outside [1, 64] points."""
    from .keypoints_util import generate_smplx_to_coco_mappings
    names = keypoint_names()
    if isinstance(select, str):
        if select != "coco":
            raise ValueError(f"select must be 'coco' or a list of point names, got {select!r}")
        return generate_smplx_to_coco_mappings(names)
    select = list(select)
    unknown = [n for n in select if n not in names]
    if unknown:
        raise ValueError(f"unknown point names {unknown}")
    if not 1 <= len(select) <= L.KP_MAX_SELECT:
        raise ValueError(f"select 1 to {L.KP_MAX_SELECT} points, got {len(select)}")
    return [names.index(n) for n in select]


def _aligned(t):
    t = t.detach().float().contiguous()
    return t.clone() if t.data_ptr() % 16 else t


def keypoints(pose, model, betas=None, transl=None, select="coco"):
    """Joints and face landmarks of a full-skeleton SMPL-X forward, in one kernel and without skinning the mesh.
    pose (F, 22 | 55 | 60, 3) axis-angle CUDA tensor (22: hands / jaw / eyes identity; 60: joints past 54 ignored);
    betas None, up to 10 values (every frame) or a CUDA tensor (F, <= 10) (one row per frame); transl (F,3) CUDA tensor or
    None; select 'coco' or a list of names from ``keypoint_names()``.  model: ``SmplxBodyModel`` (landmarks are its
    pose-blended, skinned vertices) or ``SyntheticBodyModel(skeleton='full')`` (rigid children of the head).
    Returns (F, n, 3) fp32 CUDA."""
    if not isinstance(model, (SmplxBodyModel, SyntheticBodyModel)):
        raise TypeError("keypoints needs a SmplxBodyModel or a SyntheticBodyModel(skeleton='full')")
    model.check_keypoints()
    sel = keypoint_indices(select)
    for name, t in (("pose", pose), ("transl", transl), ("betas", betas)):
        if torch.is_tensor(t) and not t.is_cuda or (name == "pose" and not torch.is_tensor(pose)):
            raise RuntimeError(f"keypoints: {name} must be a CUDA tensor -- there is no CPU fallback")
    if transl is not None and not torch.is_tensor(transl):
        raise RuntimeError("keypoints: transl must be a CUDA tensor -- there is no CPU fallback")
    if pose.dim() != 3 or pose.shape[1] not in (22, SMPLX_NUM_JOINTS, 60) or pose.shape[2] != 3:
        raise ValueError(f"keypoints: pose must be (F, 22 | 55 | 60, 3), got {tuple(pose.shape)}")
    F, dev = pose.shape[0], pose.device
    for name, t in (("transl", transl), ("betas", betas)):
        if torch.is_tensor(t) and t.device != dev:
            raise ValueError(f"keypoints: {name} is on {t.device}, pose on {dev}")
    if transl is not None and tuple(transl.shape) != (F, 3):
        raise ValueError(f"keypoints: transl must be ({F}, 3), got {tuple(transl.shape)}")
    pack = model.keypoint_pack(dev)
    B = pack.n_betas
    per_frame, b = 0, None
    if torch.is_tensor(betas) and betas.dim() == 2:
        if betas.shape[0] != F or betas.shape[1] > min(SMPLX_NUM_BETAS, B):
            raise ValueError(f"keypoints: per-frame betas must be ({F}, <= {min(SMPLX_NUM_BETAS, B)}), got {tuple(betas.shape)}")
        b = _aligned(torch.nn.functional.pad(betas.detach().float(), (0, B - betas.shape[1])))
        per_frame = 1
    elif betas is not None:
        v = (betas.detach().float().cpu().numpy() if torch.is_tensor(betas) else np.asarray(betas, dtype=np.float32)).reshape(-1)
        if v.shape[0] > min(SMPLX_NUM_BETAS, B):
            raise ValueError(f"keypoints: at most {min(SMPLX_NUM_BETAS, B)} betas, got {v.shape[0]}")
        b = torch.from_numpy(np.pad(v, (0, B - v.shape[0]))).to(dev)
    pose = _aligned(pose)
    if transl is not None:
        transl = _aligned(transl)
    out = torch.empty((F, len(sel), 3), dtype=torch.float32, device=dev)
    sel_c = (C.c_int32 * len(sel))(*sel)
    with L.on_device(pose):
        L.check(L.lib().tik_body_keypoints(C.byref(pack.c), L.ptr(pose), pose.shape[1], L.ptr(b), per_frame, L.ptr(transl),
                                           sel_c, len(sel), F, L.ptr(out), L.stream_ptr(dev)))
    return out


FIT_PRIOR_WEIGHT = 1e-3          # 1 rad away from init_pose costs as much as a 3 cm miss of one point at weight 1


def _fit_args(fn, target, model, init_pose, transl, weights, prior_weight, n_iter, select, **tensors):
    """The argument checks that fit_keypoints and fit_keypoints_shape share (``fn`` names the caller in the messages;
    ``tensors`` are further optional inputs that must be CUDA tensors on target's device when they are tensors).
    Returns the selection, the frame count, the device, the keypoint pack and the device inputs."""
    if not isinstance(model, (SmplxBodyModel, SyntheticBodyModel)):
        raise TypeError(f"{fn} needs a SmplxBodyModel or a SyntheticBodyModel(skeleton='full')")
    model.check_keypoints()
    sel = keypoint_indices(select)
    n = len(sel)
    opt = [("transl", transl), *tensors.items(), ("weights", weights)]
    for name, t in [("target", target), ("init_pose", init_pose), *opt]:
        if torch.is_tensor(t) and not t.is_cuda or (name in ("target", "init_pose") and not torch.is_tensor(t)):
            raise RuntimeError(f"{fn}: {name} must be a CUDA tensor -- there is no CPU fallback")
    if transl is not None and not torch.is_tensor(transl):
        raise RuntimeError(f"{fn}: transl must be a CUDA tensor -- there is no CPU fallback")
    if target.dim() != 3 or target.shape[1] != n or target.shape[2] != 3:
        raise ValueError(f"{fn}: target must be (F, {n}, 3) for the {n} selected points, got {tuple(target.shape)}")
    F, dev = target.shape[0], target.device
    if tuple(init_pose.shape) not in ((F, 22, 3), (F, 66)):
        raise ValueError(f"{fn}: init_pose must be ({F}, 22, 3) or ({F}, 66), got {tuple(init_pose.shape)}")
    for name, t in [("init_pose", init_pose), *opt]:
        if torch.is_tensor(t) and t.device != dev:
            raise ValueError(f"{fn}: {name} is on {t.device}, target on {dev}")
    if transl is not None and tuple(transl.shape) != (F, 3):
        raise ValueError(f"{fn}: transl must be ({F}, 3), got {tuple(transl.shape)}")
    prior_weight = float(prior_weight)
    if not (prior_weight > 0 and np.isfinite(prior_weight)):
        raise ValueError(f"{fn}: prior_weight must be positive and finite, got {prior_weight}")
    if int(n_iter) != n_iter or n_iter < 0:
        raise ValueError(f"{fn}: n_iter must be a non-negative integer, got {n_iter}")
    w, w_per_frame = None, 0
    if torch.is_tensor(weights) and weights.dim() == 2:
        if tuple(weights.shape) != (F, n):
            raise ValueError(f"{fn}: per-frame weights must be ({F}, {n}), got {tuple(weights.shape)}")
        w, w_per_frame = _aligned(weights), 1
    elif weights is not None:
        v = (weights.detach().float().cpu().numpy() if torch.is_tensor(weights) else np.asarray(weights, dtype=np.float32)).reshape(-1)
        if v.shape[0] != n:
            raise ValueError(f"{fn}: weights must have {n} values (one per selected point), got {v.shape[0]}")
        if not (v >= 0).all():
            raise ValueError(f"{fn}: weights must be non-negative")
        w = torch.from_numpy(np.ascontiguousarray(v)).to(dev)
    return dict(sel=sel, n=n, F=F, dev=dev, pack=model.keypoint_pack(dev), w=w, w_per_frame=w_per_frame,
                y=_aligned(target), pose0=_aligned(init_pose.reshape(F, 22, 3)),
                tr=None if transl is None else _aligned(transl), prior_weight=prior_weight)


def _betas_vector(fn, betas, B, dev):
    """One beta vector (at most min(10, B) values) -> (B,) fp32 on dev, zero-padded."""
    v = (betas.detach().float().cpu().numpy() if torch.is_tensor(betas) else np.asarray(betas, dtype=np.float32)).reshape(-1)
    if v.shape[0] > min(SMPLX_NUM_BETAS, B):
        raise ValueError(f"{fn}: at most {min(SMPLX_NUM_BETAS, B)} betas, got {v.shape[0]}")
    return torch.from_numpy(np.pad(v, (0, B - v.shape[0]))).to(dev)


def fit_keypoints(target, model, init_pose, betas=None, transl=None, select="coco", weights=None,
                  prior_weight=FIT_PRIOR_WEIGHT, n_iter=10, fit_transl=True):
    """Body poses whose ``keypoints`` hit ``target``: per frame, ``n_iter`` Levenberg-Marquardt steps (one
    ``tik_fit_keypoints`` launch, one warp per frame) on

        E = sum_k w_k |keypoints(pose, model, betas, transl, select)[k] - target[k]|^2 + prior_weight |pose - init_pose|^2

    over the rotations of joints 0..21 and, with ``fit_transl``, the translation.  target (F, n, 3) CUDA tensor, n the
    length of ``select`` ('coco' or names from ``keypoint_names()``); model, betas: as ``keypoints``; init_pose (F, 22, 3)
    or (F, 66) (``run_inference``'s rows), the start and the prior's centre; transl (F, 3) CUDA tensor or None (zero):
    the start (``fit_transl``) or the fixed translation; weights None (all 1), n non-negative values for every frame or a
    CUDA tensor (F, n); prior_weight > 0.  A point that the observation does not really have (e.g. the face points that
    ``moveai_to_coco`` synthesises from the ears) should get weight 0.  E never increases; a frame whose initial E is not
    finite comes back unchanged with cost NaN.
    Returns {"poses": (F, 22, 3), "transl": (F, 3), "cost_init": (F,), "cost": (F,)}, fp32 CUDA tensors."""
    a = _fit_args("fit_keypoints", target, model, init_pose, transl, weights, prior_weight, n_iter, select, betas=betas)
    sel, n, F, dev, pack = a["sel"], a["n"], a["F"], a["dev"], a["pack"]
    w, w_per_frame, y, pose0, tr, prior_weight = a["w"], a["w_per_frame"], a["y"], a["pose0"], a["tr"], a["prior_weight"]
    B = pack.n_betas
    per_frame, b = 0, None
    if torch.is_tensor(betas) and betas.dim() == 2:
        if betas.shape[0] != F or betas.shape[1] > min(SMPLX_NUM_BETAS, B):
            raise ValueError(f"fit_keypoints: per-frame betas must be ({F}, <= {min(SMPLX_NUM_BETAS, B)}), got {tuple(betas.shape)}")
        b = _aligned(torch.nn.functional.pad(betas.detach().float(), (0, B - betas.shape[1])))
        per_frame = 1
    elif betas is not None:
        b = _betas_vector("fit_keypoints", betas, B, dev)
    poses = torch.empty((F, 22, 3), dtype=torch.float32, device=dev)
    transl_out = torch.empty((F, 3), dtype=torch.float32, device=dev)
    cost = torch.empty((F, 2), dtype=torch.float32, device=dev)
    sel_c = (C.c_int32 * n)(*sel)
    with L.on_device(dev):
        L.check(L.lib().tik_fit_keypoints(C.byref(pack.c), L.ptr(y), L.ptr(w), w_per_frame, L.ptr(pose0), L.ptr(b), per_frame,
                                          L.ptr(tr), int(bool(fit_transl)), sel_c, n, prior_weight, int(n_iter), F,
                                          L.ptr(poses), L.ptr(transl_out), L.ptr(cost), L.stream_ptr(dev)))
    return {"poses": poses, "transl": transl_out, "cost_init": cost[:, 0], "cost": cost[:, 1]}


# Weight of |beta|^2 in fit_keypoints_shape.  Betas are whitened PCA coefficients (unit variance over the population), so
# this is a Gaussian prior on the shape.  At 1e-3 a shape 1 sigma from the mean costs as much as a 3 cm miss of one point
# in one frame (as FIT_PRIOR_WEIGHT does for 1 rad of pose): over a clip of hundreds of frames the data decides the shape,
# and on a clip of a few frames the prior still keeps directions the keypoints do not see near the mean.
FIT_SHAPE_PRIOR_WEIGHT = 1e-3


def fit_keypoints_shape(target, model, init_pose, lengths=None, betas=None, transl=None, select="coco", weights=None,
                        prior_weight=FIT_PRIOR_WEIGHT, shape_prior_weight=FIT_SHAPE_PRIOR_WEIGHT, n_iter=10,
                        fit_transl=True):
    """One body shape per sequence and a pose per frame whose ``keypoints`` hit ``target``: per sequence s,
    ``n_iter`` Levenberg-Marquardt steps (``tik_fit_keypoints_shape``) on

        E_s = sum_{f in s} [ sum_k w_k |keypoints(pose_f, model, beta_s, transl_f)[k] - target_f[k]|^2
                             + prior_weight |pose_f - init_pose_f|^2 ] + shape_prior_weight |beta_s|^2

    over beta_s (the model's shape coefficients, 10 for both model kinds), the rotations of joints 0..21 of every frame and,
    with ``fit_transl``, the translations.  target, model, init_pose, transl, select, weights, prior_weight, n_iter: as
    ``fit_keypoints`` (frames of every sequence packed back to back); lengths: host ints, the frame count of each sequence
    (sum = F), None for one sequence; betas: the start of the shape -- None (the mean shape, 0), one vector for every
    sequence or a CUDA tensor (S, <= 10); shape_prior_weight > 0, the weight of the prior centred on the mean shape.  E_s
    never increases; a sequence whose initial E_s is not finite comes back unchanged with cost NaN.  A sequence's results
    do not depend on the other sequences of the call.
    Returns {"poses": (F, 22, 3), "transl": (F, 3), "betas": (S, B), "cost_init": (S,), "cost": (S,)}, fp32 CUDA
    tensors."""
    from .inference import sequence_tables
    a = _fit_args("fit_keypoints_shape", target, model, init_pose, transl, weights, prior_weight, n_iter, select,
                  betas=betas)
    sel, n, F, dev, pack = a["sel"], a["n"], a["F"], a["dev"], a["pack"]
    B = pack.n_betas
    shape_prior_weight = float(shape_prior_weight)
    if not (shape_prior_weight > 0 and np.isfinite(shape_prior_weight)):
        raise ValueError(f"fit_keypoints_shape: shape_prior_weight must be positive and finite, got {shape_prior_weight}")
    if lengths is None:
        lengths = [F] if F > 0 else []
    lengths = [int(k) for k in lengths]
    if F == 0 and not lengths:
        fs = np.zeros(1, dtype=np.int64)
    else:
        fs = sequence_tables(lengths, 1, -1, 1)[0]
    S = len(lengths)
    if int(fs[-1]) != F:
        raise ValueError(f"fit_keypoints_shape: lengths sum to {int(fs[-1])}, target has {F} frames")
    if torch.is_tensor(betas) and betas.dim() == 2:
        if betas.shape[0] != S or betas.shape[1] > min(SMPLX_NUM_BETAS, B):
            raise ValueError(f"fit_keypoints_shape: per-sequence betas must be ({S}, <= {min(SMPLX_NUM_BETAS, B)}), "
                             f"got {tuple(betas.shape)}")
        b = _aligned(torch.nn.functional.pad(betas.detach().float(), (0, B - betas.shape[1])))
    elif betas is not None:
        b = _betas_vector("fit_keypoints_shape", betas, B, dev).expand(S, B).contiguous()
    else:
        b = None
    poses = torch.empty((F, 22, 3), dtype=torch.float32, device=dev)
    transl_out = torch.empty((F, 3), dtype=torch.float32, device=dev)
    betas_out = torch.empty((S, B), dtype=torch.float32, device=dev)
    cost = torch.empty((S, 2), dtype=torch.float32, device=dev)
    if F == 0:
        return {"poses": poses, "transl": transl_out, "betas": betas_out, "cost_init": cost[:, 0], "cost": cost[:, 1]}
    frame_start = torch.from_numpy(fs).to(dev)
    sel_c = (C.c_int32 * n)(*sel)
    nbytes = C.c_int64()
    L.check(L.lib().tik_fit_keypoints_shape_workspace_bytes(C.byref(pack.c), n, int(bool(fit_transl)), F, S,
                                                             C.byref(nbytes)))
    ws = torch.empty(max(1, nbytes.value), dtype=torch.uint8, device=dev)
    with L.on_device(dev):
        L.check(L.lib().tik_fit_keypoints_shape(
            C.byref(pack.c), L.ptr(a["y"]), L.ptr(a["w"]), a["w_per_frame"], L.ptr(a["pose0"]), L.ptr(a["tr"]),
            int(bool(fit_transl)), L.ptr(frame_start), S, L.ptr(b), shape_prior_weight, sel_c, n, a["prior_weight"],
            int(n_iter), F, L.ptr(ws), nbytes.value, L.ptr(poses), L.ptr(transl_out), L.ptr(betas_out), L.ptr(cost),
            L.stream_ptr(dev)))
    return {"poses": poses, "transl": transl_out, "betas": betas_out, "cost_init": cost[:, 0], "cost": cost[:, 1]}


def run_smpl_keypoints(data, smplx_models, device, apply_trans=True, apply_root_rot=True, apply_shape=True):
    """COCO-17 keypoints (F, 17, 3) numpy of the same ``data`` dict and flags as ``run_smpl_inference``: equal to
    ``smplx_joints_to_coco(run_smpl_inference(...))`` on a full-skeleton model, from one ``keypoints`` launch (the body of
    the reference's amass_data_to_3d_keypoints, inference.py:70-79).  Works for every ``SmplxBodyModel`` and for
    synthetic full-skeleton models."""
    model = smplx_models[str(data["gender"])]
    poses = torch.as_tensor(full_pose_from_amass(data["poses"], SMPLX_NUM_JOINTS)).to(device)
    if not apply_root_rot:
        poses[:, 0] = 0
    transl = torch.as_tensor(np.asarray(data["trans"], dtype=np.float32)).to(device) if apply_trans else None
    betas = np.asarray(data["betas"])[:SMPLX_NUM_BETAS] if apply_shape else None
    return keypoints(poses, model, betas, transl, "coco").cpu().numpy()


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
