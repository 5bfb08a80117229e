"""PoseRegressor / IKPoseTrainer with the reference's API on top of the CUDA engine.

Mirrors reference pose_trainer.py:66-133 (PoseRegressor) and :136-144 (IKPoseTrainer.forward and the
``regressor.`` state_dict prefix used by Lightning checkpoints, inference.py:136).  Training
(pose_trainer.py:146-260) is out of scope: the CUDA path is eval-only.
"""
import argparse
import os

import numpy as np
import torch
import torch.nn as nn

from . import engine
from .st_gcn import StgConfig, StgGcn18, StgLayerConfig, _ComputeDtypeMixin, _default_dtype

# (in_channels, out_channels, temporal_stride) of the eight blocks; the first in_channels is hparams.kps_channel
_BLOCKS = [(None, 64, 1), (64, 64, 1), (64, 128, 2), (128, 128, 1), (128, 128, 1), (128, 128, 2), (128, 256, 2),
           (256, 256, 2)]


def default_hparams(**over):
    """The argparse defaults of reference pose_trainer.py:204-218."""
    hp = dict(lr=1e-4, win_size=9, bs=256, kps_channel=3, graph_layout="coco", max_hop=2, dilation=1,
              keypoint_format="coco", n_out_joints=22, n_out_channels=3)
    hp.update(over)
    return argparse.Namespace(**hp)


class PoseRegressor(engine.EngineHolder, nn.Module, _ComputeDtypeMixin):
    def __init__(self, hparams):
        super().__init__()
        self.graph_cfg = dict(layout=hparams.graph_layout, strategy="uniform", max_hop=hparams.max_hop,
                              dilation=hparams.dilation)
        layers = [StgLayerConfig(in_channels=hparams.kps_channel if ci is None else ci, out_channels=co,
                                 temporal_stride=s, is_residual=True) for ci, co, s in _BLOCKS]
        self.backbone = StgGcn18(config=StgConfig(layers=layers, temporal_kernel_size=3), graph_cfg=self.graph_cfg)
        self.pose_dim = 22 * 3
        self.pose_regressor = nn.Sequential(nn.Linear(17 * 256, 512), nn.LeakyReLU(), nn.Dropout(0.7),
                                            nn.Linear(512, self.pose_dim))
        self.compute_dtype = _default_dtype()
        self.chunk_clips = None
        self.use_cuda_graph = os.environ.get("TIK_CUDA_GRAPH", "0") == "1"   # replay the launch sequence as one graph
        self.weight_check = None           # None = engine default ('version'); 'content': see engine.Engine
        # low_latency: batches of a few clips (N * T' <= 32, e.g. one streaming window) run as ONE persistent cooperative
        # kernel in fp32 (engine.LatencyPlan) instead of the launch-bound 19-25 kernel throughput plan
        self.low_latency = os.environ.get("TIK_LOW_LATENCY", "0") == "1"
        self._engine = None

    def _head(self):
        return self.pose_regressor[0], self.pose_regressor[1].negative_slope, self.pose_regressor[3]

    def plan_for(self, N, T):
        if self._engine is None:
            self._engine = engine.Engine(self.backbone, self._head)
        self._engine.weight_check = self.weight_check or self._engine.weight_check
        if self._use_latency_plan(N, T):
            return self._engine.latency_plan(N, T)
        return self._engine.plan(self.compute_dtype, N, T, self.chunk_clips)

    def session(self, N, T):
        """A bound forward for a serving loop: resolves the plan for (N, T) ONCE (weights are folded as they are now) and
        returns ``run(x) -> poses`` that only launches -- none of ``forward``'s per-call checks (eval / device / shape
        checks, the cache stamp over ~160 tensors: ~50 us of Python, as much as the kernel at batch 1).  ``x`` must be a
        contiguous fp32 CUDA tensor of exactly (N, T, V, C) on the model's device and current stream; make a new session
        after changing weights.  Uses the latency plan when ``low_latency`` is set and the batch fits it."""
        if self.training:
            raise NotImplementedError("PoseRegressor.session: eval-mode inference only")
        plan = self.plan_for(N, T)
        if isinstance(plan, engine.LatencyPlan):
            return plan.run
        if self.use_cuda_graph:
            return plan.run_graphed
        return lambda x: plan.run(x)[0]

    def _use_latency_plan(self, N, T):
        return (self.low_latency and self.backbone.A.size(0) == 1 and len(self.backbone.st_gcn_networks) >= 2
                and N * self.backbone.out_frames(T) <= engine.LatencyPlan.LIMIT_ROWS)

    def forward(self, x, init_pose=None, n_iter=3):
        """x (N, T, V, C) -> {'poses': (N, T', 66)} axis-angle, joint-major (reference pose_trainer.py:94-133).
        ``init_pose`` / ``n_iter`` belong to the reference's commented-out iterative 6-D head and are ignored
        there as well."""
        engine.require_cuda_eval(self, x, "PoseRegressor")
        x = self.backbone._check_input(x)
        N, T = x.shape[0], x.shape[1]
        if N == 0:
            return {"poses": x.new_zeros((0, self.backbone.out_frames(T), self.pose_dim))}
        plan = self.plan_for(N, T)
        if isinstance(plan, engine.LatencyPlan):
            return {"poses": plan.run(x)}
        poses = plan.run_graphed(x) if self.use_cuda_graph else plan.run(x)[0]
        return {"poses": poses}


    def forward_windows(self, seq, win_frames, offset=0, stride=1, root=None, n_windows=None, lengths=None):
        """Sliding-window inference over ONE sequence without materialising the windows.

        seq (F, V, C) CUDA fp32.  Window n, frame t is seq[clamp(n*stride + t + offset, 0, F-1)], optionally
        root-centred on 0.5*(kp[root[0]] + kp[root[1]]).  `offset=-(win//2)` with one window per frame reproduces
        InferenceDataset / sample_window (reference data_amass.py:18-42,221-236); `offset=0` gives plain
        [n, n+win) windows (BASELINE config 5).  Returns {'poses': (n_windows, T', 66)}.

        lengths (host ints, sum = F): seq packs several sequences back to back and every one gets the windows it would
        get on its own (n_windows must be None), clamped to its own frames; they come out in sequence order, in one
        pass, equal bit for bit to torch.cat of the per-sequence calls (inference.sequence_tables)."""
        engine.require_cuda_eval(self, seq, "PoseRegressor.forward_windows")
        if seq.dim() != 3 or seq.shape[1] != self.backbone.A.size(1) or seq.shape[2] != self.backbone.st_gcn_networks[0].in_channels:
            raise ValueError(f"expected a (F, {self.backbone.A.size(1)}, C) sequence, got {tuple(seq.shape)}")
        seq = seq.detach().float().contiguous()
        F = seq.shape[0]
        V = seq.shape[1]
        if root is not None and (len(root) != 2 or not all(0 <= int(r) < V for r in root)):
            raise ValueError(f"root must be a pair of keypoint indices in [0, {V}), got {root!r}")
        if F < 1 or int(stride) < 1 or int(win_frames) < 1:
            raise ValueError("forward_windows needs a non-empty sequence, stride >= 1 and win_frames >= 1")
        tables = None
        if lengths is not None:
            from .inference import sequence_tables
            if n_windows is not None:
                raise ValueError("forward_windows: n_windows follows from lengths; pass one or the other")
            win_frames, offset, stride = int(win_frames), int(offset), int(stride)
            tables = np.stack(sequence_tables(lengths, win_frames, offset, stride))
            if int(tables[0, -1]) != F:
                raise ValueError(f"lengths sum to {int(tables[0, -1])} frames, the packed sequence has {F}")
            n_windows = int(tables[1, -1])
        elif n_windows is None:
            n_windows = F if offset < 0 else max(0, (F - win_frames - offset) // stride + 1)
        if n_windows == 0:
            return {"poses": seq.new_zeros((0, self.backbone.out_frames(win_frames), self.pose_dim))}
        plan = self.plan_for(n_windows, win_frames)
        if tables is None:
            return {"poses": plan.run_windows(seq, n_windows, offset, stride, root)}
        return {"poses": plan.run_seq_windows(seq, torch.from_numpy(tables).to(seq.device), n_windows, offset, stride, root)}


class IterativePoseRegressor(engine.EngineHolder, nn.Module, _ComputeDtypeMixin):
    """The HMR-style iterative 6-D head the reference keeps commented out (pose_trainer.py:53-64 definition, :108-126
    forward; SURVEY.md 8f row 4), as a first-class model on the same backbone:

        pred = init_pose;  n_iter times:  xc = fc2(fc1(cat[features, pred]));  pred = decpose(xc) + pred
        rotmats = rot6d_to_rotmat(pred);  poses = rotation_matrix_to_angle_axis(rotmats)

    (dropouts are identities in eval; the reference text has no activation between fc1 and fc2).  Everything runs in
    libtik.so: the backbone plan, the three Linear layers as tensor-core / fp32 implicit GEMMs (`tik_rowgemm`; the
    concatenation is two K slabs, the 132 pose columns zero-padded to 192) and the conversion kernels.  The reference
    loads SPIN's mean pose for `init_pose`; here it defaults to the 6-D identity and can be passed in."""

    NPOSE = 22 * 6
    NPAD = 192                      # pose columns / decpose rows padded to the 64-wide MMA granule

    def __init__(self, hparams, init_pose=None, channel=512):
        super().__init__()
        self.graph_cfg = dict(layout=hparams.graph_layout, strategy="uniform", max_hop=hparams.max_hop,
                              dilation=hparams.dilation)
        layers = [StgLayerConfig(in_channels=hparams.kps_channel if ci is None else ci, out_channels=co,
                                 temporal_stride=s, is_residual=True) for ci, co, s in _BLOCKS]
        self.backbone = StgGcn18(config=StgConfig(layers=layers, temporal_kernel_size=3), graph_cfg=self.graph_cfg)
        self.fc1 = nn.Linear(17 * 256 + self.NPOSE, channel)
        self.drop1 = nn.Dropout()
        self.fc2 = nn.Linear(channel, channel)
        self.drop2 = nn.Dropout()
        self.decpose = nn.Linear(channel, self.NPOSE)
        nn.init.xavier_uniform_(self.decpose.weight, gain=0.01)
        if init_pose is None:
            init_pose = torch.tensor([1.0, 0.0, 0.0, 1.0, 0.0, 0.0]).repeat(22)
        self.register_buffer("init_pose", torch.as_tensor(init_pose, dtype=torch.float32).reshape(1, self.NPOSE))
        self.compute_dtype = _default_dtype()
        self.chunk_clips = None
        self.weight_check = None
        self.use_cuda_graph = True          # the iterative head's launches are replayed as one CUDA graph
        self._engine = None
        self._packed = None
        self._head_state = None

    def _head_weights(self):
        """fc1 / fc2 / decpose in the compute dtype, padded as the GEMM kernels want them; cached per parameter version."""
        ps = [self.fc1.weight, self.fc1.bias, self.fc2.weight, self.fc2.bias, self.decpose.weight, self.decpose.bias]
        stamp = (self.compute_dtype,) + tuple((t.data_ptr(), t._version) for t in ps)
        if self._packed is None or self._packed[0] != stamp:
            _, tdt = engine.resolve_dtype(self.compute_dtype)
            feat = 17 * 256
            w1 = self.fc1.weight.detach()
            w1 = torch.cat([w1, w1.new_zeros(w1.shape[0], self.NPAD - self.NPOSE)], dim=1)          # (512, 4352 + 192)
            assert w1.shape[1] == feat + self.NPAD
            w3 = self.decpose.weight.detach()
            w3 = torch.cat([w3, w3.new_zeros(self.NPAD - self.NPOSE, w3.shape[1])], dim=0)          # (192, 512)
            b3 = torch.cat([self.decpose.bias.detach(), self.decpose.bias.new_zeros(self.NPAD - self.NPOSE)])
            self._packed = (stamp, w1.to(tdt).contiguous(), self.fc1.bias.detach().float().reshape(1, -1).contiguous(),
                            self.fc2.weight.detach().to(tdt).contiguous(), self.fc2.bias.detach().float().reshape(1, -1).contiguous(),
                            w3.to(tdt).contiguous(), b3.float().reshape(1, -1).contiguous())
        return self._packed[1:]

    def forward(self, x, init_pose=None, n_iter=3):
        """x (N, T, V, C) -> {'poses': (N, T', 66) axis-angle, 'rotmats': (N*T', 22, 3, 3)}."""
        from . import geometry, ops
        engine.require_cuda_eval(self, x, "IterativePoseRegressor")
        x = self.backbone._check_input(x)
        N, T = x.shape[0], x.shape[1]
        Tp = self.backbone.out_frames(T)
        if N == 0:
            return {"poses": x.new_zeros((0, Tp, 66)), "rotmats": x.new_zeros((0, 22, 3, 3))}
        if self._engine is None:
            self._engine = engine.Engine(self.backbone)
        self._engine.weight_check = self.weight_check or self._engine.weight_check
        plan = self._engine.plan(self.compute_dtype, N, T, self.chunk_clips)
        _, feat = plan.run(x, want_feat=True)                               # (N, T', 17*256) in the compute dtype
        M = N * Tp
        init = (self.init_pose if init_pose is None else init_pose.to(x.device).float().reshape(-1, self.NPOSE)).expand(M, -1)
        pred = self._run_head(feat.view(1, M, -1), init, int(n_iter))
        rotmats = geometry.rot6d_to_rotmat(pred.reshape(-1, 6)).view(M, 22, 3, 3)
        poses = geometry.rotation_matrix_to_angle_axis(rotmats.reshape(-1, 3, 3)).reshape(N, Tp, 66)
        return {"poses": poses, "rotmats": rotmats}

    def _run_head(self, feat, init, n_iter):
        """pred = init; n_iter x { pred += decpose(fc2(fc1(cat[features, pred]))) } on preallocated buffers: the nine
        `tik_rowgemm` launches and the small element-wise updates of one forward are captured ONCE per (rows, n_iter,
        weights) as a CUDA graph and replayed (stable addresses: libtik re-uses its prepared launches; no allocator
        traffic; one host call instead of ~20)."""
        from . import ops
        M = feat.shape[1]
        w1, b1, w2, b2, w3, b3 = self._head_weights()
        key = (M, n_iter, feat.dtype, feat.device, torch.cuda.current_stream(feat.device).cuda_stream, id(w1))
        st = self._head_state
        if st is None or st["key"] != key:
            dev, dt = feat.device, feat.dtype
            st = {"key": key, "feat": torch.empty_like(feat), "init": torch.empty((M, self.NPOSE), device=dev),
                  "pred": torch.empty((M, self.NPOSE), device=dev), "slab": torch.zeros((1, M, self.NPAD), dtype=dt, device=dev),
                  "h1": torch.empty((1, M, w1.shape[0]), dtype=dt, device=dev), "h2": torch.empty((1, M, w2.shape[0]), dtype=dt, device=dev),
                  "d": torch.empty((M, self.NPOSE), device=dev), "graph": None, "weights": (w1, b1, w2, b2, w3, b3)}

            def body():
                st["pred"].copy_(st["init"])
                for _ in range(n_iter):
                    st["slab"][0, :, : self.NPOSE] = st["pred"]
                    ops.rowgemm([(st["feat"], 1, 0), (st["slab"], 1, 0)], w1, b1, 1, 1, M, out=st["h1"])
                    ops.rowgemm([(st["h1"], 1, 0)], w2, b2, 1, 1, M, out=st["h2"])
                    ops.rowgemm([(st["h2"], 1, 0)], w3, b3, 1, 1, M, out_layout="rows_f32", c_out_valid=self.NPOSE, out=st["d"])
                    st["pred"].add_(st["d"])

            st["feat"].copy_(feat)
            st["init"].copy_(init)
            body()                                                # eager warm-up (lazy init, prepared launches)
            if self.use_cuda_graph:
                torch.cuda.current_stream(feat.device).synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    body()
                st["graph"] = graph
            st["body"] = body
            self._head_state = st
            if not self.use_cuda_graph:
                return st["pred"].clone()
        st["feat"].copy_(feat)
        st["init"].copy_(init)
        if st["graph"] is not None:
            st["graph"].replay()
        else:
            st["body"]()
        return st["pred"].clone()


class IKPoseTrainer(engine.EngineHolder, nn.Module, _ComputeDtypeMixin):
    """Inference-side stand-in for the reference LightningModule (pose_trainer.py:136-144): same attribute
    names (``hparams``, ``regressor``, ``device``), same forward, loads Lightning checkpoints."""

    def __init__(self, hparams=None):
        super().__init__()
        self.hparams = hparams if hparams is not None else default_hparams()
        self.regressor = PoseRegressor(self.hparams)
        self.compute_dtype = _default_dtype()

    @property
    def device(self):
        return next(self.parameters()).device

    def forward(self, keypoints_3d):
        return self.regressor(keypoints_3d)

    @classmethod
    def load_from_checkpoint(cls, path, map_location=None):
        """Reads a pytorch_lightning checkpoint written by the reference trainer (inference.py:136): a dict with
        ``state_dict`` (keys prefixed ``regressor.``) and the pickled hparams."""
        ckpt = torch.load(path, map_location=map_location or "cpu", weights_only=False)
        hp = ckpt.get("hparams", ckpt.get("hyper_parameters", None))
        if isinstance(hp, dict):
            hp = default_hparams(**hp)
        model = cls(hp)
        sd = {k: v for k, v in ckpt["state_dict"].items() if k.startswith("regressor.")}
        model.load_state_dict(sd, strict=True)
        return model

    def training_step(self, *a, **k):
        raise NotImplementedError("training is out of scope for the CUDA inference path (reference pose_trainer.py:146)")
