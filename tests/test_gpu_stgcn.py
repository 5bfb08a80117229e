"""ST-GCN IK forward on the GPU (through libtik.so) vs the oracle / reference-generated goldens."""
import numpy as np
import pytest
import torch

import packed_emulator
from oracle import stgcn_port as sp, synth

pytestmark = pytest.mark.gpu

TOL_F32 = 1e-4          # north_star tolerance for the fp32 path
TOL_BF16_ABS = 0.08     # stated bf16 tolerance on 'poses' (output RMS ~1.3 rad): max-abs
TOL_BF16_RMS = 0.02     # and RMS error


def _model(seed=0, dtype="fp32", cuda=True):
    from temporal_inverse_kinematics_b200.pose_regressor import PoseRegressor, default_hparams
    m = PoseRegressor(default_hparams()).eval()
    sd = synth.make_regressor_state(sp.build_adjacency("coco", "uniform", 2, 1), seed=seed)
    m.load_state_dict(sd, strict=True)
    return (m.cuda() if cuda else m).set_compute_dtype(dtype), sd


@pytest.mark.parametrize("tag", ["t9", "t64", "t13", "t1", "t128"])
def test_fp32_matches_reference_golden(golden, tag):
    g = golden("stgcn.npz")
    m, sd = _model()
    assert synth.state_checksum(sd) == float(g["state_checksum"])
    n, t, seed = [int(v) for v in g[f"{tag}_shape"]]
    y = m(synth.make_clips(n, t, seed=seed).cuda())["poses"].cpu().numpy()
    assert y.shape == g[f"{tag}_poses"].shape
    assert np.abs(y - g[f"{tag}_poses"]).max() < TOL_F32
    feat = m.backbone(synth.make_clips(n, t, seed=seed).cuda()).cpu().numpy()
    assert np.abs(feat.reshape(-1)[:2048] - g[f"{tag}_feat_head"]).max() < TOL_F32


@pytest.mark.parametrize("n,t,chunk", [(5, 9, 2), (3, 64, None), (7, 20, 3), (64, 9, None)])
def test_fp32_matches_oracle_with_chunking(n, t, chunk):
    m, sd = _model()
    m.chunk_clips = chunk
    x = synth.make_clips(n, t, seed=n * 100 + t)
    y = m(x.cuda())["poses"].cpu()
    want = sp.regressor_forward(sd, x)["poses"]
    assert float((y - want).abs().max()) < TOL_F32


@pytest.mark.parametrize("n,t,chunk", [(4, 64, None), (5, 9, 2), (3, 13, None), (2, 128, 1), (40, 16, 16)])
def test_bf16_within_stated_tolerance(n, t, chunk):
    m, sd = _model(dtype="bf16")
    m.chunk_clips = chunk
    x = synth.make_clips(n, t, seed=n * 100 + t)
    y = m(x.cuda())["poses"].cpu()
    want = sp.regressor_forward(sd, x)["poses"]
    err = (y - want).abs()
    assert float(err.max()) < TOL_BF16_ABS, float(err.max())
    assert float(err.pow(2).mean().sqrt()) < TOL_BF16_RMS
    # the tensor-core path must agree with a bf16-rounding emulation of the same packed algebra much more tightly
    from temporal_inverse_kinematics_b200 import engine
    mc, _ = _model(dtype="bf16", cuda=False)
    emu = packed_emulator.forward(engine.PackedNet(mc.backbone, mc._head(), "bf16"), x)
    assert float((y - emu).abs().max()) < 0.05


def test_dance_config1(golden):
    """BASELINE.json configs[0]: dance_contemporary.npz windows, win_size 9."""
    g = golden("dance.npz")
    m, sd = _model()
    assert synth.state_checksum(sd) == float(g["state_checksum"])
    names = [str(s) for s in g["joint_3d_names"]]
    wins = sp.inference_windows(sp.moveai_to_coco(g["joints_3d"], names), 9).astype(np.float32)
    y = m(torch.from_numpy(wins).cuda())["poses"].cpu().numpy()
    assert y.shape == (231, 1, 66)
    assert np.abs(y - g["poses"]).max() < TOL_F32
    y1 = torch.cat([m(torch.from_numpy(wins[i:i + 1]).cuda())["poses"] for i in range(0, 231, 23)]).cpu().numpy()
    assert np.abs(y1 - g["poses"][::23]).max() < TOL_F32              # batch 1, as configs[0] runs it


@pytest.mark.parametrize("dtype,tol", [("fp32", TOL_F32), ("bf16", 0.15)])
def test_backbone_variants(golden, dtype, tol):
    """K=3 partitions (distance / spatial), temporal kernel 5, a block without residual."""
    from temporal_inverse_kinematics_b200.st_gcn import StgConfig, StgGcn18, StgLayerConfig
    g = golden("stgcn_variants.npz")
    layers = [(3, 64, 1, True), (64, 64, 2, True), (64, 128, 1, True)]
    cases = [("distance", 2, 3, layers, 5, 77, 10, "distance2_feat"), ("spatial", 1, 3, layers, 5, 77, 10, "spatial1_feat"),
             ("spatial", 2, 3, layers, 5, 77, 10, "spatial2_feat"),
             ("uniform", 2, 5, [(3, 64, 1, False), (64, 64, 1, True), (64, 128, 2, True)], 6, 78, 11, "kt5_feat")]
    for strategy, max_hop, kt, lay, seed, xseed, t, key in cases:
        graph_cfg = dict(layout="coco", strategy=strategy, max_hop=max_hop, dilation=1)
        bb = StgGcn18(StgConfig([StgLayerConfig(*l) for l in lay], kt), graph_cfg).eval()
        bb.load_state_dict(synth.make_backbone_state(sp.build_adjacency("coco", strategy, max_hop, 1), lay, kt=kt, seed=seed, prefix=""))
        bb = bb.cuda().set_compute_dtype(dtype)
        f = bb(synth.make_clips(2, t, seed=xseed).cuda()).cpu().numpy()
        assert f.shape == g[key].shape
        assert np.abs(f - g[key]).max() < tol, (key, np.abs(f - g[key]).max())


@pytest.mark.parametrize("K", [1, 3])
def test_graph_conv_module_matches_reference(golden, K):
    from temporal_inverse_kinematics_b200.st_gcn import ConvTemporalGraphical
    g = golden("stgcn_variants.npz")
    m = ConvTemporalGraphical(8, 16, K).eval()
    m.load_state_dict({"conv.weight": torch.from_numpy(g[f"gconv{K}_w"]), "conv.bias": torch.from_numpy(g[f"gconv{K}_b"])})
    m = m.cuda()
    y, A = m(torch.from_numpy(g[f"gconv{K}_x"]).cuda(), torch.from_numpy(g[f"gconv{K}_A"]).cuda())
    assert y.shape == g[f"gconv{K}_y"].shape and y.is_contiguous()
    assert np.abs(y.cpu().numpy() - g[f"gconv{K}_y"]).max() < TOL_F32


@pytest.mark.parametrize("cin,cout,stride,residual,dtype,tol", [
    (3, 64, 1, True, "fp32", TOL_F32), (64, 64, 1, True, "fp32", TOL_F32), (64, 128, 2, True, "fp32", TOL_F32),
    (64, 64, 1, False, "fp32", TOL_F32), (64, 128, 2, True, "bf16", 0.06), (128, 128, 1, True, "bf16", 0.06)])
def test_block_module_matches_oracle(cin, cout, stride, residual, dtype, tol):
    from temporal_inverse_kinematics_b200.st_gcn import StGcnBlock
    A = sp.build_adjacency("coco", "uniform", 2, 1)
    sd_all = synth.make_backbone_state(A, [(cin, cout, stride, residual)], kt=3, seed=9, prefix="")
    sd = {k[len("st_gcn_networks.0."):]: v for k, v in sd_all.items() if k.startswith("st_gcn_networks.0.")}
    blk = StGcnBlock(cin, cout, (3, 1), stride, residual=residual).eval()
    blk.load_state_dict(sd, strict=True)
    blk = blk.cuda().set_compute_dtype(dtype)
    x = torch.from_numpy(np.random.RandomState(4).standard_normal((3, cin, 11, 17)).astype(np.float32))
    Ah = torch.from_numpy(A.astype(np.float32)) * sd_all["edge_importance.0"]
    y, _ = blk(x.cuda(), Ah.cuda())
    with torch.no_grad():
        want = sp.st_gcn_block(x, Ah, sd_all, "st_gcn_networks.0.", cin, cout, stride, residual)
    assert y.shape == want.shape
    assert float((y.cpu() - want).abs().max()) < tol


def test_weight_update_invalidates_cache():
    m, sd = _model()
    x = synth.make_clips(2, 9, seed=1).cuda()
    y0 = m(x)["poses"].clone()
    with torch.no_grad():
        m.pose_regressor[3].bias.add_(1.0)
    y1 = m(x)["poses"]
    assert float((y1 - y0 - 1.0).abs().max()) < 1e-5


def test_errors_surface_as_exceptions():
    m, _ = _model()
    with pytest.raises(ValueError):
        m(torch.zeros(2, 9, 16, 3).cuda())                            # wrong node count
    assert m(torch.zeros(0, 9, 17, 3).cuda())["poses"].shape == (0, 1, 66)


def test_cuda_graph_replay_matches_eager():
    m, sd = _model(dtype="bf16")
    x = synth.make_clips(6, 32, seed=5).cuda()
    y0 = m(x)["poses"].clone()
    m.use_cuda_graph = True
    y1 = m(x)["poses"]
    y2 = m(x)["poses"]
    assert torch.equal(y0, y1) and torch.equal(y1, y2) and y1.data_ptr() != y2.data_ptr()
    x2 = synth.make_clips(6, 32, seed=6).cuda()                          # new address -> new graph
    want = sp.regressor_forward(sd, x2.cpu())["poses"]
    assert float((m(x2)["poses"].cpu() - want).abs().max()) < TOL_BF16_ABS


def test_run_inference_matches_reference_pipeline(golden):
    """inference.run_inference on dance_contemporary.npz: GPU windowing + root-centring + model vs the reference's
    host pipeline outputs (tests/golden/dance.npz)."""
    from temporal_inverse_kinematics_b200 import inference, keypoints_util
    from temporal_inverse_kinematics_b200.pose_regressor import IKPoseTrainer
    g = golden("dance.npz")
    names = [str(s) for s in g["joint_3d_names"]]
    seq = keypoints_util.moveai_to_coco(g["joints_3d"], names)
    assert np.array_equal(seq, g["coco_seq"])
    tr = IKPoseTrainer().eval()
    sd = synth.make_regressor_state(sp.build_adjacency("coco", "uniform", 2, 1), seed=0)
    tr.regressor.load_state_dict(sd, strict=True)
    tr = tr.cuda()
    out = inference.run_inference(tr, seq)
    assert out.shape == (231, 66)
    assert np.abs(out - g["poses"][:, 0]).max() < TOL_F32


@pytest.mark.parametrize("win,offset,stride", [(9, -4, 1), (16, 0, 1), (13, 0, 3), (64, -32, 5)])
def test_forward_windows_equals_materialised_windows(win, offset, stride):
    m, sd = _model()
    F = 150
    seq = synth.make_clips(1, F, seed=33)[0]                          # (F,17,3)
    n_windows = F if offset < 0 else (F - win - offset) // stride + 1
    idx = (torch.arange(n_windows)[:, None] * stride + torch.arange(win)[None, :] + offset).clamp(0, F - 1)
    wins = seq[idx]                                                   # (n, win, 17, 3)
    wins = wins - 0.5 * (wins[:, :, 11] + wins[:, :, 12])[:, :, None, :]
    want = m(wins.cuda())["poses"]
    got = m.forward_windows(seq.cuda(), win, offset=offset, stride=stride, root=(11, 12), n_windows=n_windows)["poses"]
    assert got.shape == want.shape
    assert float((got - want).abs().max()) < 1e-5


def test_window_mean_matches_reference_loop():
    from temporal_inverse_kinematics_b200.inference import window_mean
    F, hw, D = 23, 2, 5
    preds = torch.randn(F, 2 * hw + 1, D, device="cuda")
    p = preds.cpu().numpy()
    lists = [[] for _ in range(F)]
    for i in range(F):                                               # the reference's accumulation, inference.py:56-67
        for o in range(-hw, hw + 1):
            if 0 <= i + o < F:
                lists[i + o].append(p[i, o + hw])
    want = np.array([np.mean(np.array(l), axis=0) for l in lists])
    assert np.abs(window_mean(preds, hw).cpu().numpy() - want).max() < 1e-6
    assert torch.equal(window_mean(preds, 0), preds[:, 0])


@pytest.mark.parametrize("win,offset,stride", [(9, -4, 1), (64, -32, 5), (30, 0, 2)])
def test_bf16_forward_windows_equals_materialised_windows(win, offset, stride):
    """Window mode of the fused first-block kernel (frames gathered from the resident sequence with edge clamping and
    root-centring inside the kernel) vs the same kernel fed materialised windows.  The two differ only in where the
    root is subtracted (before vs inside the folded data_bn + aggregation), i.e. by fp32 rounding ahead of the bf16
    hi/lo split."""
    m, sd = _model(dtype="bf16")
    F = 150
    seq = synth.make_clips(1, F, seed=34)[0]
    n_windows = F if offset < 0 else (F - win - offset) // stride + 1
    idx = (torch.arange(n_windows)[:, None] * stride + torch.arange(win)[None, :] + offset).clamp(0, F - 1)
    wins = seq[idx]
    wins = wins - 0.5 * (wins[:, :, 11] + wins[:, :, 12])[:, :, None, :]
    want = m(wins.cuda())["poses"]
    got = m.forward_windows(seq.cuda(), win, offset=offset, stride=stride, root=(11, 12), n_windows=n_windows)["poses"]
    assert got.shape == want.shape
    assert float((got - want).abs().max()) < 0.03
    ref = sp.regressor_forward(sd, wins)["poses"]
    assert float((got.cpu() - ref).abs().max()) < TOL_BF16_ABS


@pytest.mark.parametrize("dtype,chunk,low_latency", [("fp32", None, False), ("bf16", 3, False), ("fp32", None, True)])
def test_batch_is_window_mode_with_stride_T(dtype, chunk, low_latency):
    """A batch of N clips of T frames is window mode over its own N*T frames with stride T, offset 0 and no root: the
    stem kernels load the same addresses either way, so model(x) equals forward_windows bit for bit (fp32 stem kernel,
    fused first block over several chunks, latency plan)."""
    from temporal_inverse_kinematics_b200 import engine
    n, t = 8, 40
    m, _ = _model(dtype=dtype)
    m.chunk_clips, m.low_latency = chunk, low_latency
    assert isinstance(m.plan_for(n, t), engine.LatencyPlan) == low_latency
    x = synth.make_clips(n, t, seed=55).cuda()
    want = m(x)["poses"]
    got = m.forward_windows(x.reshape(n * t, 17, 3), t, offset=0, stride=t, root=None, n_windows=n)["poses"]
    assert torch.equal(got, want)


@pytest.mark.parametrize("switch", ["TIK_NO_STEM_BLOCK", "TIK_NO_TS", "TIK_NO_FUSED_GCN", "TIK_NO_TCN_HALO"])
def test_bf16_kernel_variants_agree(monkeypatch, switch):
    """Every specialised tensor-core kernel has a more general one behind it (first block: stem + temporal conv;
    halo / weight-stationary temporal conv: per-tap TS kernel, then the SS-mode kernel; fused graph conv, the 256-channel
    one included: aggregate + channel GEMM).  Both routes must meet the stated bf16 tolerance against the oracle and stay
    close to each other."""
    x = synth.make_clips(6, 40, seed=21)
    m, sd = _model(dtype="bf16")
    fast = m(x.cuda())["poses"].cpu()
    monkeypatch.setenv(switch, "1")
    m2, _ = _model(dtype="bf16")                                      # plans are built at first use: new model, new plan
    slow = m2(x.cuda())["poses"].cpu()
    want = sp.regressor_forward(sd, x)["poses"]
    assert float((fast - want).abs().max()) < TOL_BF16_ABS
    assert float((slow - want).abs().max()) < TOL_BF16_ABS
    assert float((fast - slow).abs().max()) < 0.06


@pytest.mark.parametrize("dtype,n,t", [("bf16", 300, 64), ("bf16", 37, 128), ("bf16", 5, 9), ("fp32", 40, 64)])
def test_serpentine_order_is_bit_identical(monkeypatch, dtype, n, t):
    """Consecutive kernels walk the clips in opposite directions (LaunchOpts::rev, csrc/plan.cu): a pure re-ordering of
    independent tiles, so the poses must not change by a single bit."""
    x = synth.make_clips(n, t, seed=77).cuda()
    m, _ = _model(dtype=dtype)
    monkeypatch.setenv("TIK_SERPENTINE", "0")
    base = m(x)["poses"].clone()
    monkeypatch.setenv("TIK_SERPENTINE", "1")
    assert torch.equal(m(x)["poses"], base)


@pytest.mark.parametrize("n,t", [(1, 1), (1, 2), (2, 11), (1, 12), (2, 13), (3, 25), (7, 33), (2, 61), (1, 65), (2, 95),
                                 (1, 100), (2, 126), (1, 127), (1, 129), (1, 190), (1, 191), (1, 200), (1, 256), (33, 16)])
def test_bf16_edge_shapes(n, t):
    """Tile-boundary cases of the specialised kernels: min(T, 13) output frames per tile in the fused first block, G row
    groups of L+2 rows per tile in the halo temporal conv (long clips cut into segments of L frames, the last one ragged
    when no divisor of T fits), odd tile counts in the paired 64-channel graph conv, single clips and single frames
    (tests/tools/shape_sweep.py has the long list; tests/test_gpu_plan_blocks.py checks each block against fp64)."""
    m, sd = _model(dtype="bf16")
    x = synth.make_clips(n, t, seed=1000 * n + t)
    want = sp.regressor_forward(sd, x)["poses"]
    got = m(x.cuda())["poses"].cpu()
    assert got.shape == want.shape and torch.isfinite(got).all()
    assert float((got - want).abs().max()) < TOL_BF16_ABS


@pytest.mark.parametrize("n,t", [(1, 64), (2, 64), (1, 9), (7, 9), (32, 9), (1, 13), (3, 33), (4, 128), (1, 1), (2, 200)])
def test_latency_plan_matches_reference_path(n, t):
    """One persistent cooperative kernel for a handful of clips (csrc/latency.cu): fp32, so the 1e-4 parity bar of the
    fp32 path applies, and it must agree with the multi-launch fp32 plan to rounding."""
    m, sd = _model()
    x = synth.make_clips(n, t, seed=7000 + 10 * n + t)
    want = sp.regressor_forward(sd, x)["poses"]
    multi = m(x.cuda())["poses"].cpu()
    m.low_latency = True
    plan = m.plan_for(n, t)
    from temporal_inverse_kinematics_b200 import engine
    assert isinstance(plan, engine.LatencyPlan) and plan.launches(n) == 1
    got = m(x.cuda())["poses"].cpu()
    assert got.shape == want.shape
    assert float((got - want).abs().max()) < TOL_F32
    assert float((got - multi).abs().max()) < 4e-5      # fp32 FMA (latency plan) vs 3xTF32 tensor-core GEMMs: each ~1e-5 from the reference
    # batches above the head's 32-row limit fall back to the throughput plan
    big = synth.make_clips(40, t, seed=1)
    assert not isinstance(m.plan_for(40, t), engine.LatencyPlan) or 40 * m.backbone.out_frames(t) <= 32
    assert m(big.cuda())["poses"].shape[0] == 40


def test_latency_plan_dance_batch1_and_windows(golden):
    """configs[0] through the latency plan (231 windows of 9 frames, batch 1) and window mode of configs[4]."""
    g = golden("dance.npz")
    m, sd = _model()
    m.low_latency = True
    names = [str(s) for s in g["joint_3d_names"]]
    wins = sp.inference_windows(sp.moveai_to_coco(g["joints_3d"], names), 9).astype(np.float32)
    y1 = torch.cat([m(torch.from_numpy(wins[i:i + 1]).cuda())["poses"] for i in range(0, 231, 11)]).cpu().numpy()
    assert np.abs(y1 - g["poses"][::11]).max() < TOL_F32
    F = 150
    seq = synth.make_clips(1, F, seed=33)[0]
    idx = (torch.arange(4)[:, None] * 3 + torch.arange(64)[None, :] - 32).clamp(0, F - 1)
    w = seq[idx]
    w = w - 0.5 * (w[:, :, 11] + w[:, :, 12])[:, :, None, :]
    want = sp.regressor_forward(sd, w)["poses"]
    got = m.forward_windows(seq.cuda(), 64, offset=-32, stride=3, root=(11, 12), n_windows=4)["poses"].cpu()
    assert float((got - want).abs().max()) < TOL_F32


def test_session_is_the_same_forward():
    """model.session(N, T): the bound forward of a serving loop returns exactly what model(x) returns, on every plan."""
    x = synth.make_clips(1, 64, seed=77).cuda()
    for dtype, low, graph in (("bf16", False, False), ("bf16", False, True), ("fp32", True, False)):
        m, _ = _model(dtype=dtype)
        m.low_latency, m.use_cuda_graph = low, graph
        want = m(x)["poses"]
        run = m.session(1, 64)
        assert torch.equal(run(x), want) and torch.equal(run(x), want)


def test_rotation_aware_window_mean():
    """SURVEY 8f row 2 option: rotations are averaged as rotations.  Two predictions of (almost) the same half-turn
    written as +(pi - e) and -(pi - e) about one axis average to ~zero rotation in the reference's euclidean mean and to
    the half-turn in rotation mode; for tightly clustered predictions both modes agree."""
    from oracle import geometry_port as gp
    from temporal_inverse_kinematics_b200.inference import window_mean
    F, hw = 9, 1
    rs = np.random.RandomState(3)
    base = rs.standard_normal((F, 22, 3)).astype(np.float32) * 0.4
    preds = np.repeat(base[:, None], 2 * hw + 1, axis=1) + rs.standard_normal((F, 3, 22, 3)).astype(np.float32) * 1e-3
    # frame f receives window i = f - o at slot o + hw; make every contribution to a frame a small perturbation of base[f]
    p = np.zeros_like(preds)
    for i in range(F):
        for o in range(-hw, hw + 1):
            if 0 <= i + o < F:
                p[i, o + hw] = base[i + o] + rs.standard_normal((22, 3)).astype(np.float32) * 1e-3
    t = torch.from_numpy(p.reshape(F, 3, 66)).cuda()
    e = window_mean(t, hw).cpu().numpy()
    r = window_mean(t, hw, mode="rotation").cpu().numpy()
    assert np.abs(e - r).max() < 5e-3 and np.abs(r.reshape(F, 22, 3) - base).max() < 5e-3
    # half-turn about z seen from both sides
    q = np.zeros((F, 3, 22, 3), dtype=np.float32)
    q[:, 0, :, 2] = np.pi - 0.05
    q[:, 1, :, 2] = -(np.pi - 0.05)
    q[:, 2, :, 2] = np.pi - 0.05
    t = torch.from_numpy(q.reshape(F, 3, 66)).cuda()
    e = window_mean(t, hw).cpu().numpy().reshape(F, 22, 3)
    r = window_mean(t, hw, mode="rotation").cpu().numpy().reshape(F, 22, 3)
    Rr = gp.batch_rodrigues(r[2:-2].reshape(-1, 3)).reshape(-1, 3, 3)
    half_turn = np.diag([-1.0, -1.0, 1.0])
    assert np.abs(Rr - half_turn).max() < 0.12            # within the 0.05 rad spread of the inputs
    assert np.abs(e[2:-2, :, 2]).max() < 1.2              # the euclidean mean collapses towards zero rotation
    with pytest.raises(ValueError):
        window_mean(t, hw, mode="geodesic")
