"""Ragged sequence batches: forward_windows(lengths=...), window_mean(lengths=...) and run_inference_batch.

CPU: the sequence tables against brute-force enumeration, and the host-side argument checks of the C entry points
and of the Python wrappers.  GPU: a ragged batch equals the per-sequence calls bit for bit (fp32 and bf16, throughput
and latency plans, sequences straddling chunks), agrees with materialised windows, leaves the memory around its
outputs alone and replays as a CUDA graph."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import stgcn_port as sp, synth
from temporal_inverse_kinematics_b200 import _lib
from temporal_inverse_kinematics_b200.inference import sequence_tables, window_mean

INVALID = _lib._H["TIK_ERR_INVALID"]
LENGTHS = [1, 3, 8, 9, 10, 231, 517]
SHUFFLED = [231, 1, 517, 9, 3, 10, 8]
WINDOWS = [(9, -4, 1), (64, -32, 5), (16, 0, 1)]


def _brute_tables(lengths, win, offset, stride):
    fs, ws = [0], [0]
    for F in lengths:
        n = 0
        if offset < 0:
            n = F
        else:
            while n * stride + offset + win <= F:             # window n fits inside the sequence
                n += 1
        fs.append(fs[-1] + F)
        ws.append(ws[-1] + n)
    return np.array(fs), np.array(ws)


@pytest.mark.parametrize("offset", [-4, -1, 0, 2])
@pytest.mark.parametrize("stride", [1, 3, 5])
def test_sequence_tables_match_enumeration(offset, stride):
    for lengths in ([1], [1, 1, 1], LENGTHS, SHUFFLED, [2, 15, 16, 17, 40]):
        for win in (1, 9, 16):
            fs, ws = sequence_tables(lengths, win, offset, stride)
            bfs, bws = _brute_tables(lengths, win, offset, stride)
            assert fs.dtype == np.int64 and ws.dtype == np.int64
            assert np.array_equal(fs, bfs) and np.array_equal(ws, bws), (lengths, win, offset, stride)


def test_sequence_tables_reject_bad_lengths():
    for bad in ([], [3, 0, 2], [4, -1]):
        with pytest.raises(ValueError):
            sequence_tables(bad, 9, -4, 1)
    with pytest.raises(ValueError, match="sequence 1"):
        sequence_tables([3, 0], 9, -4, 1)


def _expect_invalid(rc, needle):
    assert rc == INVALID
    msg = _lib.lib().tik_last_error().decode()
    assert needle in msg, msg


def test_c_entry_points_reject_bad_arguments_on_the_host():
    """Every check runs before any device work: fake device pointers are never dereferenced, no GPU is needed."""
    lib = _lib.lib()
    fake = C.c_void_p(256)
    win = _lib.TikWindowing(100, -4, 1, 11, 12)
    seqs = _lib.TikSeqBatch(2, 256, 512)
    for fn, extra in ((lib.tik_stgcn_plan_run_seq_windows, (fake, None, None)), (lib.tik_stgcn_latency_run_seq_windows, (fake, None))):
        _expect_invalid(fn(None, fake, C.byref(win), C.byref(seqs), 10, *extra), "null plan")
        _expect_invalid(fn(None, fake, None, C.byref(seqs), 10, *extra), "null windowing")
        _expect_invalid(fn(None, fake, C.byref(win), None, 10, *extra), "null windowing or sequence batch")
        _expect_invalid(fn(None, fake, C.byref(win), C.byref(_lib.TikSeqBatch(0, 256, 512)), 10, *extra), "n_seqs")
        _expect_invalid(fn(None, fake, C.byref(win), C.byref(_lib.TikSeqBatch(2, None, 512)), 10, *extra), "table")
        _expect_invalid(fn(None, fake, C.byref(win), C.byref(_lib.TikSeqBatch(2, 256, None)), 10, *extra), "table")
        _expect_invalid(fn(None, fake, C.byref(win), C.byref(seqs), -1, *extra), "n_windows")
        for bad in (_lib.TikWindowing(100, -4, 0, 11, 12), _lib.TikWindowing(0, -4, 1, 11, 12)):
            _expect_invalid(fn(None, fake, C.byref(bad), C.byref(seqs), 10, *extra), "stride")
        _expect_invalid(fn(None, fake, C.byref(_lib.TikWindowing(100, -4, 1, 11, -1)), C.byref(seqs), 10, *extra), "root")
    wm = lib.tik_window_mean
    s = None
    _expect_invalid(wm(None, 10, 5, 66, fake, 2, 1, 0, fake, s), "null")
    _expect_invalid(wm(fake, 10, 5, 66, None, 2, 1, 0, fake, s), "null")
    _expect_invalid(wm(fake, 10, 5, 66, fake, 2, 1, 0, None, s), "null")
    _expect_invalid(wm(fake, 10, 5, 66, fake, 0, 1, 0, fake, s), "n_seqs")
    _expect_invalid(wm(fake, -1, 5, 66, fake, 2, 1, 0, fake, s), "shape")
    _expect_invalid(wm(fake, 10, 5, 66, fake, 2, -1, 0, fake, s), "h_w_size")
    _expect_invalid(wm(fake, 10, 5, 66, fake, 2, 3, 0, fake, s), "2h+1")
    _expect_invalid(wm(fake, 10, 5, 64, fake, 2, 1, _lib.MEAN_ROTATION, fake, s), "divisible by 3")
    _expect_invalid(wm(fake, 10, 5, 66, fake, 2, 1, 7, fake, s), "mode")


def test_python_argument_errors_without_a_device():
    from temporal_inverse_kinematics_b200.inference import run_inference_batch
    preds = torch.zeros(10, 5, 66)
    with pytest.raises(ValueError, match="sum to 9"):
        window_mean(preds, 2, lengths=[4, 5])
    with pytest.raises(ValueError):
        window_mean(preds, 2, lengths=[10, 0])
    with pytest.raises(ValueError):
        window_mean(preds, 2, lengths=[11, -1])
    with pytest.raises(ValueError, match="predictions per window"):
        window_mean(preds, 3, lengths=[10])
    with pytest.raises(ValueError, match="divisible by 3"):
        window_mean(torch.zeros(10, 5, 64), 1, mode="rotation", lengths=[10])
    assert run_inference_batch(None, []) == []
    with pytest.raises(ValueError, match="sequence 1"):
        run_inference_batch(None, [np.zeros((5, 17, 3)), np.zeros((0, 17, 3))])


# ------------------------------------------------------------------------------------------------------------ GPU

def _model(dtype="fp32", seed=0):
    from temporal_inverse_kinematics_b200.pose_regressor import PoseRegressor, default_hparams
    m = PoseRegressor(default_hparams()).eval()
    m.load_state_dict(synth.make_regressor_state(sp.build_adjacency("coco", "uniform", 2, 1), seed=seed), strict=True)
    return m.cuda().set_compute_dtype(dtype)


def _packed(lengths, seed=0):
    return torch.cat([synth.make_clips(1, F, seed=seed + 7 * F)[0] for F in lengths])


def _per_sequence(m, seq, lengths, win, offset, stride):
    outs, f0 = [], 0
    for F in lengths:
        outs.append(m.forward_windows(seq[f0:f0 + F], win, offset=offset, stride=stride, root=(11, 12))["poses"])
        f0 += F
    return torch.cat(outs)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("win,offset,stride", WINDOWS)
@pytest.mark.parametrize("chunk", [5, None])
def test_ragged_forward_windows_equals_per_sequence_calls(dtype, win, offset, stride, chunk):
    m = _model(dtype)
    m.chunk_clips = chunk
    for lengths in (LENGTHS, SHUFFLED):
        seq = _packed(lengths).cuda()
        want = _per_sequence(m, seq, lengths, win, offset, stride)
        got = m.forward_windows(seq, win, offset=offset, stride=stride, root=(11, 12), lengths=lengths)["poses"]
        assert got.shape == want.shape
        assert torch.equal(got, want), float((got - want).abs().max())


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,tol", [("fp32", 1e-5), ("bf16", 0.03)])
@pytest.mark.parametrize("win,offset,stride", WINDOWS)
def test_ragged_forward_windows_equals_materialised_windows(dtype, tol, win, offset, stride):
    m = _model(dtype)
    lengths = SHUFFLED
    seq = _packed(lengths)
    fs, ws = sequence_tables(lengths, win, offset, stride)
    clips = []
    for s, F in enumerate(lengths):                                   # the CPU index oracle
        n = torch.arange(int(ws[s + 1] - ws[s]))
        idx = int(fs[s]) + (n[:, None] * stride + torch.arange(win)[None, :] + offset).clamp(0, F - 1)
        clips.append(seq[idx])
    wins = torch.cat(clips)
    wins = wins - 0.5 * (wins[:, :, 11] + wins[:, :, 12])[:, :, None, :]
    want = m(wins.cuda())["poses"]
    got = m.forward_windows(seq.cuda(), win, offset=offset, stride=stride, root=(11, 12), lengths=lengths)["poses"]
    assert got.shape == want.shape
    assert float((got - want).abs().max()) < tol


@pytest.mark.gpu
def test_latency_plan_ragged_equals_per_sequence_latency_runs():
    from temporal_inverse_kinematics_b200 import engine
    m = _model("fp32")
    m.low_latency = True
    for lengths, (win, offset, stride) in (([1, 3, 8, 9, 10], (9, -4, 1)),    # 31, 21 and 4 windows: one launch each ([20, 3, 31, 1, 10], (16, 0, 1)),
                                           ([1, 2, 1], (64, -32, 5))):
        seq = _packed(lengths, seed=5).cuda()
        n = int(sequence_tables(lengths, win, offset, stride)[1][-1])
        assert isinstance(m.plan_for(n, win), engine.LatencyPlan)
        want = _per_sequence(m, seq, lengths, win, offset, stride)
        got = m.forward_windows(seq, win, offset=offset, stride=stride, root=(11, 12), lengths=lengths)["poses"]
        assert torch.equal(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("Tp,h", [(5, 2), (9, 4), (3, 1), (1, 0), (5, 0)])
def test_ragged_window_mean_equals_per_sequence(Tp, h):
    lengths = [1, 2, 3, 17, 1, 4, 60]                                # length 1 and lengths below 2h+1
    g = torch.Generator().manual_seed(Tp * 10 + h)
    preds = (0.6 * torch.randn(sum(lengths), Tp, 66, generator=g)).cuda()
    offs = np.cumsum([0] + lengths)
    for mode in ("euclidean", "rotation"):
        got = window_mean(preds, h, mode, lengths=lengths)
        want = torch.cat([window_mean(preds[offs[k]:offs[k + 1]], h, mode) for k in range(len(lengths))])
        if h == 0:
            assert torch.equal(got, preds[:, 0])
        if mode == "euclidean":
            assert torch.equal(got, want)
        else:
            assert float((got - want).abs().max()) <= 1e-6


@pytest.mark.gpu
def test_run_inference_batch_equals_run_inference_loop(golden):
    from temporal_inverse_kinematics_b200 import inference, keypoints_util
    from temporal_inverse_kinematics_b200.pose_regressor import IKPoseTrainer, default_hparams
    g = golden("dance.npz")
    dance = keypoints_util.moveai_to_coco(g["joints_3d"], [str(s) for s in g["joint_3d_names"]])
    seqs = [synth.make_clips(1, F, seed=F)[0].numpy() for F in (1, 4, 12)] + [dance] + \
           [synth.make_clips(1, F, seed=F)[0].numpy() for F in (70, 333)]
    sd = synth.make_regressor_state(sp.build_adjacency("coco", "uniform", 2, 1), seed=0)
    for win, h, mode, dtype in ((9, 0, "euclidean", "fp32"), (9, 0, "euclidean", "bf16"), (65, 2, "euclidean", "fp32"),
                                (65, 2, "rotation", "fp32"), (65, 2, "rotation", "bf16")):
        tr = IKPoseTrainer(default_hparams(win_size=win)).eval()
        tr.regressor.load_state_dict(sd, strict=True)
        tr = tr.cuda()
        tr.regressor.set_compute_dtype(dtype)
        got = inference.run_inference_batch(tr, seqs, h_w_size=h, mean_mode=mode)
        want = [inference.run_inference(tr, s, h_w_size=h, mean_mode=mode) for s in seqs]
        assert len(got) == len(want)
        for a, b in zip(got, want):
            assert a.shape == b.shape
            if mode == "euclidean":
                assert np.array_equal(a, b)
            else:
                assert np.abs(a - b).max() <= 1e-6


def _tables(lengths, win, offset, stride):
    return torch.from_numpy(np.stack(sequence_tables(lengths, win, offset, stride))).cuda()


@pytest.mark.gpu
def test_c_abi_leaves_guard_regions_alone():
    m = _model("fp32")
    lengths, (win, offset, stride) = [5, 1, 30, 9], (9, -4, 1)
    seq = _packed(lengths).cuda()
    tab = _tables(lengths, win, offset, stride)
    n = sum(lengths)
    plan = m.plan_for(n, win)
    sentinel, G = -12345.0, 1024
    stream = _lib.stream_ptr()
    buf = torch.full((2 * G + n * 66,), sentinel, device="cuda")
    out = buf[G:G + n * 66]
    win_s = _lib.TikWindowing(n, offset, stride, 11, 12)
    seqs = _lib.TikSeqBatch(len(lengths), tab[0].data_ptr(), tab[1].data_ptr())
    _lib.check(_lib.lib().tik_stgcn_plan_run_seq_windows(plan.handle, _lib.ptr(seq), C.byref(win_s), C.byref(seqs), n,
                                                         _lib.ptr(out), None, stream))
    torch.cuda.synchronize()
    assert bool((buf[:G] == sentinel).all()) and bool((buf[G + n * 66:] == sentinel).all())
    want = m.forward_windows(seq, win, offset=offset, stride=stride, root=(11, 12), lengths=lengths)["poses"]
    assert torch.equal(out.view(n, 1, 66), want)
    for h, mode in ((0, _lib.MEAN_EUCLIDEAN), (2, _lib.MEAN_EUCLIDEAN), (2, _lib.MEAN_ROTATION)):
        preds = torch.randn(n, 5, 66, device="cuda")
        mbuf = torch.full((2 * G + n * 66,), sentinel, device="cuda")
        mout = mbuf[G:G + n * 66]
        _lib.check(_lib.lib().tik_window_mean(_lib.ptr(preds), n, 5, 66, _lib.ptr(tab[0]), len(lengths), h, mode,
                                              _lib.ptr(mout), stream))
        torch.cuda.synchronize()
        assert bool((mbuf[:G] == sentinel).all()) and bool((mbuf[G + n * 66:] == sentinel).all())
        assert bool(torch.isfinite(mout).all())
    # root keypoints are checked against the plan's node count
    bad = _lib.TikWindowing(n, offset, stride, 11, 17)
    _expect_invalid(_lib.lib().tik_stgcn_plan_run_seq_windows(plan.handle, _lib.ptr(seq), C.byref(bad), C.byref(seqs), n,
                                                              _lib.ptr(out), None, stream), "root")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_cuda_graph_replay_after_rewriting_the_input(dtype):
    from temporal_inverse_kinematics_b200.inference import packed_window_mean
    m = _model(dtype)
    lengths, (win, offset, stride), h = [7, 1, 40, 13], (65, -32, 1), 2
    n = sum(lengths)
    seq = _packed(lengths, seed=1).cuda()
    tab = _tables(lengths, win, offset, stride)
    plan = m.plan_for(n, win)

    def body():
        poses = plan.run_seq_windows(seq, tab, n, offset, stride, (11, 12))
        return packed_window_mean(poses, tab[0], h, "rotation")
    body()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = body()
    seq.copy_(_packed(lengths, seed=2).cuda())
    graph.replay()
    torch.cuda.synchronize()
    poses = m.forward_windows(seq, win, offset=offset, stride=stride, root=(11, 12), lengths=lengths)["poses"]
    assert torch.equal(out, window_mean(poses, h, "rotation", lengths=lengths))


@pytest.mark.gpu
def test_argument_errors_raise_before_any_launch():
    m = _model("fp32")
    seq = _packed([5, 6]).cuda()
    with pytest.raises(ValueError, match="sum to"):
        m.forward_windows(seq, 9, offset=-4, root=(11, 12), lengths=[5, 5])
    with pytest.raises(ValueError):
        m.forward_windows(seq, 9, offset=-4, root=(11, 12), lengths=[11, 0])
    with pytest.raises(ValueError):
        m.forward_windows(seq, 9, offset=-4, root=(11, 12), lengths=[12, -1])
    with pytest.raises(ValueError, match="n_windows"):
        m.forward_windows(seq, 9, offset=-4, root=(11, 12), lengths=[5, 6], n_windows=11)
    preds = torch.zeros(11, 1, 66, device="cuda")
    with pytest.raises(ValueError, match="sum to"):
        window_mean(preds, 0, lengths=[5, 5])
    with pytest.raises(ValueError, match="predictions per window"):
        window_mean(preds, 1, lengths=[5, 6])
    assert m.forward_windows(seq, 16, offset=0, root=(11, 12), lengths=[5, 6])["poses"].shape == (0, 1, 66)
