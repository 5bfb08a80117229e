"""Boundary checks that need no GPU: the product Graph against the reference-generated goldens, state_dict
round trips in the reference's layout (pinned by what its own modules left in tests/golden/stgcn.npz),
Lightning-style checkpoints, pickling, cache invalidation, the header-derived limits, and the independent FK
cross-check of the oracle (scipy-composed homogeneous chain)."""
import copy
import io
import os

import numpy as np
import pytest
import torch

from oracle import fk_port, fk_scipy, geometry_port as gp, ref_import, stgcn_port as sp, synth
from temporal_inverse_kinematics_b200 import _lib, engine, smpl_util
from temporal_inverse_kinematics_b200.graph import Graph
from temporal_inverse_kinematics_b200.pose_regressor import IKPoseTrainer, PoseRegressor, default_hparams
from temporal_inverse_kinematics_b200.st_gcn import StgConfig, StgGcn18, StgLayerConfig


def test_product_graph_bit_identical_to_reference(golden):
    """The class the models actually construct (not the oracle's builder): mmskeleton/ops/st_gcn/graph.py:4-133."""
    g = golden("graph.npz")
    assert len(g.files) == 48
    for key in g.files:
        layout, strategy, max_hop, dilation = key.split("|")
        gr = Graph(layout=layout, strategy=strategy, max_hop=int(max_hop), dilation=int(dilation))
        assert gr.A.dtype == g[key].dtype and gr.A.shape == g[key].shape, key
        assert np.array_equal(gr.A, g[key]), key
    A = Graph("coco", "uniform", 2, 1).A
    assert A.shape == (1, 17, 17) and int((A != 0).sum()) == 107
    # and the buffer a freshly constructed model carries is that adjacency in fp32
    m = PoseRegressor(default_hparams())
    assert torch.equal(m.backbone.A, torch.tensor(g["coco|uniform|2|1"], dtype=torch.float32))


def _reference_state(golden):
    """The state dict the reference's own PoseRegressor loaded with strict=True when tests/golden/stgcn.npz was made
    (oracle/make_golden.py); the stored checksum proves it is the same one."""
    g = golden("stgcn.npz")
    sd = synth.make_regressor_state(Graph("coco", "uniform", 2, 1).A, seed=0)
    assert synth.state_checksum(sd) == float(g["state_checksum"]), "synthetic weight stream drifted"
    return sd, g


def test_state_dict_round_trip_with_real_reference(golden):
    """pose_trainer.py:66-92: load_state_dict(strict=True) both ways in the reference's PoseRegressor layout.  The
    reference's side is what its own modules left in tests/golden/stgcn.npz: the state dict it loaded and its poses."""
    theirs, g = _reference_state(golden)
    torch.manual_seed(3)
    ours = PoseRegressor(default_hparams()).eval()
    assert list(theirs.keys()) == list(ours.state_dict().keys())
    assert all(theirs[k].shape == v.shape and theirs[k].dtype == v.dtype for k, v in ours.state_dict().items())
    ours.load_state_dict(theirs, strict=True)
    for k, v in ours.state_dict().items():
        assert torch.equal(v, theirs[k]), k
    # OUR state dict, run through the oracle port, reproduces the reference's own output (ties the three together)
    n, t, seed = [int(v) for v in g["t9_shape"]]
    y = sp.regressor_forward(ours.state_dict(), synth.make_clips(n, t, seed=seed))["poses"]
    assert float(np.abs(y.numpy() - g["t9_poses"]).max()) < 1e-5


def test_lightning_checkpoint_from_real_reference(tmp_path, golden):
    """inference.py:136: IKPoseTrainer.load_from_checkpoint on a checkpoint in the reference's own LightningModule
    layout ('regressor.' prefix, pickled hparams), carrying the state dict the reference's PoseRegressor loaded."""
    sd, _ = _reference_state(golden)
    hp = ref_import.default_hparams()
    ckpt = {"state_dict": {"regressor." + k: v for k, v in sd.items()}, "hparams": vars(hp), "epoch": 98}
    path = tmp_path / "checkpoint_epoch=98.ckpt"
    torch.save(ckpt, path)
    m = IKPoseTrainer.load_from_checkpoint(str(path))
    assert m.hparams.win_size == hp.win_size and m.hparams.graph_layout == "coco"
    for k, v in sd.items():
        assert torch.equal(m.state_dict()["regressor." + k], v), k
    # hparams stored as a Namespace (old Lightning) work as well
    ckpt["hparams"] = hp
    torch.save(ckpt, path)
    assert IKPoseTrainer.load_from_checkpoint(str(path)).hparams.max_hop == 2


def test_models_pickle_and_deepcopy_without_their_engine(tmp_path):
    m = PoseRegressor(default_hparams()).eval()
    m._engine = engine.Engine(m.backbone, m._head)                  # as after a first forward
    c = copy.deepcopy(m)
    assert c._engine is None and m._engine is not None
    buf = io.BytesIO()
    torch.save(m, buf)
    buf.seek(0)
    r = torch.load(buf, weights_only=False)
    assert r._engine is None and list(r.state_dict()) == list(m.state_dict())
    t = IKPoseTrainer()
    t.regressor._engine = engine.Engine(t.regressor.backbone, t.regressor._head)
    assert copy.deepcopy(t).regressor._engine is None
    bb = StgGcn18(StgConfig([StgLayerConfig(3, 64, 1, True)], 3), dict(layout="coco", strategy="uniform", max_hop=2, dilation=1),
                  data_bn=False)
    torch.save(bb, io.BytesIO())                                     # data_bn=False is a module-level function, not a lambda


def test_cache_stamp_covers_scalars_and_content_mode():
    m = PoseRegressor(default_hparams()).eval()
    e = engine.Engine(m.backbone, m._head)
    s0 = e._stamp_now(m.backbone, m._head())
    m.pose_regressor[1].negative_slope = 0.2
    s1 = e._stamp_now(m.backbone, m._head())
    assert s0 != s1
    m.backbone.st_gcn_networks[2].tcn[0].eps = 1e-3
    assert e._stamp_now(m.backbone, m._head()) != s1
    with torch.no_grad():
        before = e._stamp_now(m.backbone, m._head())
        m.backbone.st_gcn_networks[1].gcn.conv.weight.add_(0.1)      # autograd-visible in-place update
        assert e._stamp_now(m.backbone, m._head()) != before
    # writes through .data are invisible to the version stamp ...
    before = e._stamp_now(m.backbone, m._head())
    m.backbone.st_gcn_networks[3].tcn[2].weight.data.mul_(1.01)
    assert e._stamp_now(m.backbone, m._head()) == before
    # ... caught by the content mode, and by the explicit invalidate()
    e.weight_check = "content"
    before = e._stamp_now(m.backbone, m._head())
    m.backbone.st_gcn_networks[3].tcn[2].weight.data.mul_(1.01)
    assert e._stamp_now(m.backbone, m._head()) != before
    e._stamp = before
    e.invalidate()
    assert e._stamp is None and not e._plans and not e._packed
    m._engine = e
    m.invalidate_packed()
    e.weight_check = "bogus"
    with pytest.raises(ValueError):
        e._stamp_now(m.backbone, m._head())


def test_limits_come_from_the_header():
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "tik.h")).read()
    assert f"#define TIK_MAX_JOINTS {_lib.MAX_JOINTS}" in hdr and _lib.MAX_JOINTS == 64
    assert f"#define TIK_MAX_BLOCKS {_lib.MAX_BLOCKS}" in hdr
    assert f"#define TIK_MAX_SLABS {_lib.MAX_SLABS}" in hdr
    assert (_lib.RES_CONV, _lib.OUT_ROWS_F32) == (_lib._H["TIK_RES_CONV"], _lib._H["TIK_OUT_ROWS_F32"])


@pytest.mark.parametrize("skeleton", ["body", "full"])
def test_fk_port_agrees_with_independent_scipy_chain(skeleton):
    """fk_port (split rotation / translation, quaternion Rodrigues) vs the published homogeneous-matrix chain with
    scipy rotations (oracle/fk_scipy.py).  Both restate common/smpl_util.py:61-70 -> smplx; smplx itself is absent."""
    model = smpl_util.SyntheticBodyModel(skeleton=skeleton)
    J = len(model.parents)
    aa = synth.make_axis_angles(257, J, seed=21, scale=0.9).astype(np.float64)
    aa[0] = 0.0                                                       # rest pose
    aa[1, :, :] = 0.0
    aa[1, 0] = [0.0, 0.0, np.pi - 1e-3]                               # near-pi root rotation
    aa[2] *= 1e-7                                                     # tiny angles
    rest = model.rest_joints.astype(np.float64)
    transl = np.random.RandomState(2).standard_normal((257, 3))
    j1, R1, g1 = fk_port.fk_from_axis_angle(aa, rest, model.parents, transl)
    j2, g2 = fk_scipy.fk_homogeneous(aa, rest, model.parents, transl)
    assert np.abs(j1 - j2).max() < 1e-6 and np.abs(g1 - g2).max() < 1e-6
    assert np.abs(j1[0] - (rest + transl[0])).max() < 1e-12
    Rq = gp.batch_rodrigues(aa.reshape(-1, 3)).reshape(-1, 3, 3)
    assert np.abs(fk_scipy.rodrigues_skew(aa.reshape(-1, 3)) - Rq).max() < 1e-6


def test_device_side_moveai_remap_is_bit_identical(golden):
    """inference.py:121-133 as one gather-and-blend on the tensor's device (here: CPU tensors) vs the numpy mirror and
    the reference's own output stored in the golden."""
    from temporal_inverse_kinematics_b200 import keypoints_util as ku
    g = golden("dance.npz")
    names = [str(s) for s in g["joint_3d_names"]]
    want = ku.moveai_to_coco(g["joints_3d"], names)
    got = ku.moveai_to_coco_device(torch.from_numpy(g["joints_3d"]), names)
    assert got.dtype == torch.float32 and got.is_contiguous()
    assert np.array_equal(got.numpy(), want) and np.array_equal(want, g["coco_seq"])
