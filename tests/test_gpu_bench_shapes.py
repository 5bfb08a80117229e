"""Parity at the shapes bench.py measures (BASELINE.json configs[1..3]) and on the quantities north_star gates:
rotation matrices and joint positions, not only the axis-angle 'poses'.

The CPU oracle cannot run 4096 clips in seconds, so the GPU result of the FULL batch is compared on sampled clips
-- the first, middle and last ones (so that every persistent CTA's first and tail tiles and the last chunk are
hit) plus a seeded random set -- with the oracle run on exactly those clips."""
import numpy as np
import pytest
import torch

from oracle import fk_port, fk_scipy, stgcn_port as sp, synth

pytestmark = pytest.mark.gpu

J = 22
TOL_F32 = 1e-4                       # north_star: fp32 max-abs on rotation matrices and joint positions (and poses)
# Stated bf16 tolerances (tensor cores, fp32 accumulate, bf16 activations between kernels; untrained random weights
# give poses of 1.3 rad RMS, far harsher than a trained regressor).  Measured on B200 / emulated on CPU:
# poses 0.034 max / 0.009 RMS, rotation-matrix entries 0.033 / 0.0064, joints 0.037 m / 0.0045 m.
TOL_BF16 = {"poses": (0.08, 0.02), "rotmats": (0.08, 0.015), "joints": (0.08, 0.012)}


def _model(dtype):
    from temporal_inverse_kinematics_b200.pose_regressor import PoseRegressor, default_hparams
    m = PoseRegressor(default_hparams()).eval()
    sd = synth.make_regressor_state(sp.build_adjacency("coco", "uniform", 2, 1), seed=0)
    m.load_state_dict(sd, strict=True)
    return m.cuda().set_compute_dtype(dtype), sd


def _sample(n, k=8, extra=8, seed=0):
    idx = set(range(min(k, n))) | set(range(max(0, n // 2 - k // 2), min(n, n // 2 + k // 2))) | set(range(max(0, n - k), n))
    idx |= set(np.random.RandomState(seed).randint(0, n, extra).tolist())
    return sorted(idx)


def _gpu_solve(m, x, rest, parents):
    """poses, local rotation matrices and FK joints as bench.py's step produces them."""
    from temporal_inverse_kinematics_b200 import smpl_util
    poses = m(x)["poses"]
    joints, local_R = smpl_util.fk_body(poses.view(-1, J, 3), rest, parents, want_local=True)
    return poses, local_R.view(poses.shape[0], -1, J, 3, 3), joints.view(poses.shape[0], -1, J, 3)


def _cpu_solve(sd, x, rest, parents):
    poses = sp.regressor_forward(sd, x)["poses"].numpy()
    j, R, _ = fk_port.fk_from_axis_angle(poses.reshape(-1, J, 3).astype(np.float64), rest.astype(np.float64), parents)
    return poses, R.reshape(poses.shape[0], -1, J, 3, 3), j.reshape(poses.shape[0], -1, J, 3)


def _errs(got, want):
    e = np.abs(np.asarray(got, dtype=np.float64) - np.asarray(want, dtype=np.float64))
    return float(e.max()), float(np.sqrt((e ** 2).mean()))


@pytest.mark.parametrize("n,t", [(4096, 64), (2048, 128), (4100, 64), (300, 128)])
def test_bf16_parity_at_benchmarked_shapes(n, t):
    """configs[2] (B=4096, T=64) and the configs[3] micro-batch (2048 clips of T=128), plus ragged batches that end
    in a short chunk."""
    m, sd = _model("bf16")
    rest, parents = synth.make_rest_skeleton(), synth.SMPLX_BODY_PARENTS
    x = synth.make_clips(n, t, seed=1234)
    idx = _sample(n)
    poses, R, joints = _gpu_solve(m, x.cuda(), rest, parents)
    assert poses.shape == (n, t // 16, 66) and torch.isfinite(poses).all() and torch.isfinite(joints).all()
    w_poses, w_R, w_joints = _cpu_solve(sd, x[idx], rest, parents)
    for name, got, want in (("poses", poses, w_poses), ("rotmats", R, w_R), ("joints", joints, w_joints)):
        mx, rms = _errs(got[idx].cpu().numpy(), want)
        assert mx < TOL_BF16[name][0] and rms < TOL_BF16[name][1], (name, mx, rms)
    # the CUDA-graph replay of the same plan returns the same bits
    m.use_cuda_graph = True
    assert torch.equal(m(x.cuda())["poses"], poses)


def test_fp32_parity_config1_shapes():
    """configs[1]: B=256, T=64, fp32: poses, rotation matrices and joints within 1e-4 of the reference path for ALL
    clips (the oracle runs the full batch in about a second)."""
    m, sd = _model("fp32")
    rest, parents = synth.make_rest_skeleton(), synth.SMPLX_BODY_PARENTS
    x = synth.make_clips(256, 64, seed=1234)
    poses, R, joints = _gpu_solve(m, x.cuda(), rest, parents)
    w_poses, w_R, w_joints = _cpu_solve(sd, x, rest, parents)
    for name, got, want in (("poses", poses, w_poses), ("rotmats", R, w_R), ("joints", joints, w_joints)):
        mx, _ = _errs(got.cpu().numpy(), want)
        assert mx < TOL_F32, (name, mx)


def test_bench_dump_outputs_are_the_timed_results(tmp_path):
    """bench.py --dump-outputs writes the poses and FK joints of its last timed step; its first clips are
    synth.make_clips(seed=1234), which the oracle solves here."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--batch", "64", "--steps", "2", "--warmup", "1",
                          "--no-cpu", "--no-hbm", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    poses, joints = np.load(tmp_path / "poses.npy"), np.load(tmp_path / "joints.npy")
    assert poses.dtype == joints.dtype == np.float32 and poses.shape == (64, 4, 66) and joints.shape == (64, 4, J, 3)
    _, sd = _model("bf16")
    rest, parents = synth.make_rest_skeleton(), synth.SMPLX_BODY_PARENTS
    w_poses, _, w_joints = _cpu_solve(sd, synth.make_clips(64, 64, seed=1234), rest, parents)
    for name, got, want in (("poses", poses, w_poses), ("joints", joints, w_joints)):
        mx, rms = _errs(got, want)
        assert mx < TOL_BF16[name][0] and rms < TOL_BF16[name][1], (name, mx, rms)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_rot6d_head_variant_config1(dtype):
    """configs[1]'s second head variant (SURVEY 0.3): the commented-out iterative 6-D head + rot6d -> rotmat ->
    axis-angle; tolerances on the ROTATION MATRICES.  The Gram-Schmidt of rot6d_to_rotmat is ill-conditioned where an
    untrained head leaves a2 nearly parallel to a1 (DESIGN.md section 4), so fp32 is gated at 1e-4 on all but a
    handful of entries (<= 0.01 %; measured max 3.6e-4 over 202,752 entries at B=256) with RMS <= 1e-5; bf16 (three
    residual iterations amplify the rounding): RMS <= 0.03 (measured 0.010), <= 0.5 % of the entries above 0.1
    (measured 0.12 %, max 0.40 on an ill-conditioned row)."""
    from temporal_inverse_kinematics_b200.pose_regressor import IterativePoseRegressor, default_hparams
    sd = synth.make_iterative_state(sp.build_adjacency("coco", "uniform", 2, 1), seed=0)
    m = IterativePoseRegressor(default_hparams()).eval()
    m.load_state_dict(sd, strict=True)
    m = m.cuda().set_compute_dtype(dtype)
    n = 256 if dtype == "fp32" else 64
    x = synth.make_clips(n, 64, seed=1234)
    out = m(x.cuda())
    want = sp.iterative_regressor_forward(sd, x)
    mx, rms = _errs(out["rotmats"].cpu().numpy().reshape(-1, 3, 3), np.asarray(want["rotmats"]).reshape(-1, 3, 3))
    if dtype == "fp32":
        e = np.abs(out["rotmats"].cpu().numpy().reshape(-1) - np.asarray(want["rotmats"]).reshape(-1))
        assert rms < 1e-5 and mx < 2e-3 and float((e > TOL_F32).mean()) < 1e-4, (mx, rms, float((e > TOL_F32).mean()))
    else:
        e = np.abs(out["rotmats"].cpu().numpy().reshape(-1) - np.asarray(want["rotmats"]).reshape(-1))
        assert rms < 0.03 and float((e > 0.1).mean()) < 5e-3 and mx < 1.0, (mx, rms, float((e > 0.1).mean()))


@pytest.mark.parametrize("skeleton", ["body", "full"])
def test_fk_kernels_against_independent_scipy_chain(skeleton):
    """The FK kernels against oracle/fk_scipy.py (homogeneous chain, scipy rotations): a second, independently written
    restatement of common/smpl_util.py:61-70 -> smplx.  Joints within 1e-4 m of it."""
    from temporal_inverse_kinematics_b200 import smpl_util
    model = smpl_util.SyntheticBodyModel(skeleton=skeleton)
    Jn = len(model.parents)
    aa = synth.make_axis_angles(3001, Jn, seed=23, scale=0.8)
    aa[0] = 0.0
    aa[1, 0] = [0.0, 0.0, np.pi - 1e-3]
    transl = np.random.RandomState(3).standard_normal((3001, 3)).astype(np.float32)
    joints = smpl_util.fk_body(torch.from_numpy(aa).cuda(), model.rest_joints, model.parents, torch.from_numpy(transl).cuda())
    want, _ = fk_scipy.fk_homogeneous(aa, model.rest_joints, model.parents, transl)
    assert np.abs(joints.cpu().numpy() - want).max() < TOL_F32


def test_unaligned_views_and_bad_window_roots():
    from temporal_inverse_kinematics_b200 import geometry as G, smpl_util
    from oracle import geometry_port as gp
    aa = torch.from_numpy(synth.make_axis_angles(101, 1, seed=5).reshape(-1, 3)).cuda()
    got = G.batch_rodrigues(aa[1:])                                   # contiguous view at a 12-byte offset
    assert np.abs(got.cpu().numpy() - gp.batch_rodrigues(aa[1:].cpu().numpy())).max() < 1e-5
    R = got.view(-1, 3, 3)
    back = G.rotation_matrix_to_angle_axis(R[1:])                     # 36-byte offset
    assert back.shape == (99, 3) and torch.isfinite(back).all()
    pose = torch.from_numpy(synth.make_axis_angles(9, 22, seed=6)).cuda()
    rest, parents = synth.make_rest_skeleton(), synth.SMPLX_BODY_PARENTS
    j_full = smpl_util.fk_body(pose, rest, parents)
    assert torch.equal(smpl_util.fk_body(pose[1:], rest, parents), j_full[1:])
    m, _ = _model("bf16")
    seq = synth.make_clips(1, 40, seed=2)[0].cuda()
    for bad in [(11, 17), (-1, 12), (11,), (3, 99)]:
        with pytest.raises(ValueError):
            m.forward_windows(seq, 9, offset=-4, root=bad)


def test_data_write_needs_invalidate_or_content_check():
    """ADVICE r1: `.data` writes do not bump tensor versions; invalidate_packed() / weight_check='content' re-fold."""
    m, _ = _model("fp32")
    x = synth.make_clips(2, 9, seed=1).cuda()
    y0 = m(x)["poses"].clone()
    m.pose_regressor[3].bias.data.add_(1.0)
    m.invalidate_packed()
    y1 = m(x)["poses"].clone()
    assert float((y1 - y0 - 1.0).abs().max()) < 1e-5
    m.weight_check = "content"
    m.pose_regressor[3].bias.data.add_(1.0)
    assert float((m(x)["poses"] - y0 - 2.0).abs().max()) < 1e-5


def test_model_on_a_non_current_device_and_second_stream():
    """ADVICE r1: dispatch follows the tensors' device, not the thread's current device; each stream has its own plan."""
    m, sd = _model("bf16")
    x = synth.make_clips(3, 16, seed=4)
    want = m(x.cuda())["poses"].clone()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        got = m(x.cuda())["poses"]
    s.synchronize()
    assert torch.equal(got, want)
    assert len({k[-1] for k in m._engine._plans}) == 2               # one plan (workspace) per stream
    if torch.cuda.device_count() > 1:
        m1 = m.to("cuda:1")
        with torch.cuda.device(0):
            got1 = m1(x.to("cuda:1"))["poses"]
        assert torch.equal(got1.cpu(), want.cpu())
