"""Host side of the CUDA path: eval-mode folding of the reference parameters into packed
weights (SURVEY.md Appendix B) and cached launch plans over libtik.so.

The packed algebra, for one ST-GCN block with A^ = A * edge_importance (st_gcn_aaai18.py:128-129),
BN folded as s = gamma / sqrt(var + eps), o = beta - mean * s:

  gcn   H[n,w,t,c] = relu( sum_{k,ci} s1[c] Wg[k*Cout+c,ci] * (sum_v A^[k,v,w] X[n,v,t,ci])
                           + s1[c] * sum_k bg[k*Cout+c] * colsum_k[w] + o1[c] )        (gconv_origin.py:59-63)
  tcn   Y[n,w,t',c] = relu( sum_{dt,c'} s2[c] Wt[c,c',dt] H[n,w,s*t'+dt-pad,c'] + s2[c] bt[c] + o2[c] + R )
  res   R = X (identity) | sum_ci s3[c] Wr[c,ci] X[n,w,s*t',ci] + s3[c] br[c] + o3[c]   (st_gcn_aaai18.py:191-214)

There is no CPU or eager-PyTorch fallback: anything but eval-mode CUDA tensors raises.
"""
import ctypes as C
import operator
import os
import weakref

import torch

from . import _lib as L

BN_EPS_DEFAULT = 1e-5
_GET_VERSION, _GET_EPS, _GET_PTR = operator.attrgetter("_version"), operator.attrgetter("eps"), torch.Tensor.data_ptr
_CHECKED_DEVICES = set()
_DTYPES = {"fp32": (L.TIK_F32, torch.float32), "bf16": (L.TIK_BF16, torch.bfloat16)}


def resolve_dtype(name):
    if name not in _DTYPES:
        raise ValueError(f"compute dtype must be 'fp32' or 'bf16', got {name!r}")
    return _DTYPES[name]


def _bn_fold(bn):
    """(scale, shift) of an eval-mode BatchNorm, float64."""
    var = bn.running_var.detach().double()
    mean = bn.running_mean.detach().double()
    g = bn.weight.detach().double() if bn.weight is not None else torch.ones_like(var)
    b = bn.bias.detach().double() if bn.bias is not None else torch.zeros_like(var)
    s = g / torch.sqrt(var + bn.eps)
    return s, b - mean * s


def fold_gcn(conv_weight, conv_bias, A_hat, K, bn=None):
    """-> w (Cout, K*Cin) f64, bias table (V, Cout) f64 for the aggregate-first graph convolution."""
    KC, cin = conv_weight.shape[0], conv_weight.shape[1]
    cout = KC // K
    W = conv_weight.detach().double().reshape(K, cout, cin)               # out-channel index k*Cout+c
    bg = conv_bias.detach().double().reshape(K, cout) if conv_bias is not None else torch.zeros(K, cout, dtype=torch.float64, device=W.device)
    colsum = A_hat.detach().double().sum(dim=1)                           # (K, V): sum over v of A^[k,v,w]
    w = W.permute(1, 0, 2).reshape(cout, K * cin)
    b = torch.einsum("kc,kw->wc", bg, colsum)
    if bn is not None:
        s, o = _bn_fold(bn)
        w = w * s[:, None]
        b = b * s[None, :] + o[None, :]
    return w, b


def fold_tcn(conv, bn, res_conv=None, res_bn=None):
    """-> w (Cout, kt*Cout [+Cin]) f64, bias (Cout) f64 for temporal conv + BN (+ residual 1x1 conv + BN)."""
    Wt = conv.weight.detach().double()[..., 0]                            # (Cout, Cout, kt)
    cout, _, kt = Wt.shape
    s2, o2 = _bn_fold(bn)
    bt = conv.bias.detach().double() if conv.bias is not None else torch.zeros(cout, dtype=torch.float64, device=Wt.device)
    w = (Wt.permute(0, 2, 1) * s2[:, None, None]).reshape(cout, kt * cout)   # column dt*Cout + c'
    b = s2 * bt + o2
    wr = None
    if res_conv is not None:
        s3, o3 = _bn_fold(res_bn)
        Wr = res_conv.weight.detach().double()[:, :, 0, 0]               # (Cout, Cin)
        br = res_conv.bias.detach().double() if res_conv.bias is not None else torch.zeros(cout, dtype=torch.float64, device=Wt.device)
        wr = Wr * s3[:, None]
        b = b + s3 * br + o3
    return w, b, wr


def _raw_bn(bn):
    """TikRawBN over a BatchNorm module's own tensors (None: no BatchNorm)."""
    r = L.TikRawBN()
    if bn is None:
        return r
    f = lambda t: None if t is None else t.detach().data_ptr()
    r.weight_dev, r.bias_dev, r.mean_dev, r.var_dev, r.eps = f(bn.weight), f(bn.bias), f(bn.running_mean), f(bn.running_var), bn.eps
    return r


def raw_block(backbone, i):
    """TikRawBlock over block i's raw fp32 parameters (pointers into the module's tensors; nothing is copied)."""
    blk = backbone.st_gcn_networks[i]
    A, imp = backbone.A.detach(), backbone.edge_importance[i]
    f = lambda t: None if t is None else t.detach().data_ptr()
    for t in (blk.gcn.conv.weight, blk.tcn[2].weight, A):
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError("tik_pack_block reads contiguous fp32 parameters")
    r = L.TikRawBlock()
    r.c_in, r.c_out, r.stride, r.kt = blk.in_channels, blk.out_channels, blk.stride, blk.temporal_kernel
    r.K, r.V = A.shape[0], A.shape[1]
    r.residual = {"none": L.RES_NONE, "identity": L.RES_IDENTITY, "conv": L.RES_CONV}[blk.residual_kind]
    r.A_dev, r.importance_dev = f(A), (f(imp) if torch.is_tensor(imp) else None)
    r.gcn_w_dev, r.gcn_b_dev, r.bn1 = f(blk.gcn.conv.weight), f(blk.gcn.conv.bias), _raw_bn(blk.tcn[0])
    r.tcn_w_dev, r.tcn_b_dev, r.bn2 = f(blk.tcn[2].weight), f(blk.tcn[2].bias), _raw_bn(blk.tcn[3])
    if blk.residual_kind == "conv":
        r.res_w_dev, r.res_b_dev, r.bn_res = f(blk.residual[0].weight), f(blk.residual[0].bias), _raw_bn(blk.residual[1])
    return r


class PackedNet:
    """Device-resident packed weights + the TikNet descriptor that points at them.

    packer="host" folds with torch fp64 ops (fold_gcn / fold_tcn above); packer="device" calls the C ABI's
    tik_pack_bn / tik_pack_block on the raw parameters instead (same algebra, same rounding points; the GPU tests hold
    the two bit-identical).  Default: TIK_PACKER or "host"."""

    def __init__(self, backbone, head, dtype_name, packer=None):
        self.packer = packer or os.environ.get("TIK_PACKER", "host")
        if self.packer not in ("host", "device"):
            raise ValueError("packer must be 'host' or 'device'")
        self.dtype_name = dtype_name
        self.code, self.tdtype = resolve_dtype(dtype_name)
        dev = backbone.A.device
        self.device = dev
        self.keep = []                                                    # tensors referenced by raw pointer
        self.named = {}                                                   # same tensors by name (introspection/tests)
        net = L.TikNet()
        A = backbone.A.detach()
        K, V = A.shape[0], A.shape[1]
        blocks = list(backbone.st_gcn_networks)
        if len(blocks) > L.MAX_BLOCKS:
            raise ValueError(f"at most {L.MAX_BLOCKS} ST-GCN blocks are supported")
        cin0 = blocks[0].in_channels
        net.V, net.K, net.c_in, net.n_blocks = V, K, cin0, len(blocks)
        if isinstance(backbone.data_bn, torch.nn.BatchNorm1d):
            s0, o0 = _bn_fold(backbone.data_bn)                           # channel index v*C + c
        else:
            s0 = torch.ones(V * cin0, dtype=torch.float64, device=dev)
            o0 = torch.zeros(V * cin0, dtype=torch.float64, device=dev)
        net.in_scale_dev = self._f32(s0, "in_scale")
        net.in_shift_dev = self._f32(o0, "in_shift")
        if self.packer == "device" and isinstance(backbone.data_bn, torch.nn.BatchNorm1d):
            with L.on_device(dev):                                        # overwrite with the library's own fold
                L.check(L.lib().tik_pack_bn(C.byref(_raw_bn(backbone.data_bn)), V * cin0, L.ptr(self.named["in_scale"]),
                                            L.ptr(self.named["in_shift"]), L.stream_ptr(dev)))
        for i, blk in enumerate(blocks):
            if self.packer == "device":
                self._pack_block_device(backbone, i, net.blocks[i])
                continue
            imp = backbone.edge_importance[i]
            A_hat = A * imp.detach() if torch.is_tensor(imp) else A * imp
            b = net.blocks[i]
            b.c_in, b.c_out, b.stride, b.kt = blk.in_channels, blk.out_channels, blk.stride, blk.temporal_kernel
            wg, bg = fold_gcn(blk.gcn.conv.weight, blk.gcn.conv.bias, A_hat, K, blk.tcn[0])
            b.agg_dev = self._f32(A_hat.double(), f"b{i}.agg")
            # the stem kernel computes in fp32
            b.w_gcn_dev = self._f32(wg, f"b{i}.w_gcn") if i == 0 else self._act(wg, f"b{i}.w_gcn")
            b.b_gcn_dev = self._f32(bg, f"b{i}.b_gcn")
            res_conv = res_bn = None
            if blk.residual_kind == "conv":
                res_conv, res_bn = blk.residual[0], blk.residual[1]
            wt, bt, wr = fold_tcn(blk.tcn[2], blk.tcn[3], res_conv, res_bn)
            # tensor-core path: identity-type residuals ride through the MMA as one more K-slab against an
            # identity weight block (bf16 x 1.0 accumulated in fp32 is exact) instead of scattered epilogue loads
            fold_identity = self.code == L.TIK_BF16
            eye = torch.eye(blk.out_channels, dtype=torch.float64, device=dev)
            if blk.residual_kind == "none":
                b.res_kind = L.RES_NONE
            elif blk.residual_kind == "identity":
                if i == 0:
                    raise NotImplementedError("an identity residual on the first block is not supported by the CUDA path")
                b.res_kind = L.RES_IDENTITY
                if fold_identity:
                    wt = torch.cat([wt, eye], dim=1)
                    b.res_as_slab = 1
            elif i == 0:
                if cin0 > 8:
                    raise NotImplementedError("first-block residual convolution needs in_channels <= 8")
                b.res_kind = L.RES_STEM
                s0v, o0v = s0.view(V, cin0), o0.view(V, cin0)
                b.w_res_stem_dev = self._f32(wr[None, :, :] * s0v[:, None, :], f"b{i}.w_res_stem")  # (V, Cout, Cin)
                bt = bt[None, :] + torch.einsum("ci,vi->vc", wr, o0v)                    # (V, Cout)
                if fold_identity:
                    wt = torch.cat([wt, eye], dim=1)
                    b.res_as_slab = 1
            else:
                b.res_kind = L.RES_CONV
                wt = torch.cat([wt, wr], dim=1)
            b.w_tcn_dev = self._act(wt, f"b{i}.w_tcn")
            b.b_tcn_dev = self._f32(bt, f"b{i}.b_tcn")
        self.c_last = blocks[-1].out_channels
        if head is not None:
            lin1, slope, lin2 = head
            net.head_hidden, net.head_out = lin1.out_features, lin2.out_features
            net.leaky_slope = float(slope)
            net.w1_dev = self._act(lin1.weight.detach().double(), "w1")
            net.b1_dev = self._f32(lin1.bias.detach().double(), "b1")
            w2, b2 = lin2.weight.detach().double(), lin2.bias.detach().double()
            if self.code == L.TIK_BF16:                                    # pad rows to the 64-column MMA granule
                rows = (w2.shape[0] + 63) // 64 * 64
                w2 = torch.cat([w2, w2.new_zeros(rows - w2.shape[0], w2.shape[1])])
                b2 = torch.cat([b2, b2.new_zeros(rows - b2.shape[0])])
            net.w2_dev = self._act(w2, "w2")
            net.b2_dev = self._f32(b2, "b2")
            self.head_out = lin2.out_features
        else:
            net.head_hidden = net.head_out = 0
            self.head_out = 0
        self.net = net
        self.V, self.K, self.c_in = V, K, cin0

    def _pack_block_device(self, backbone, i, out):
        """Block i through tik_pack_block: outputs allocated here, folded by the library on the current stream."""
        lib = L.lib()
        dev = self.device
        raw = raw_block(backbone, i)
        first = 1 if i == 0 else 0
        nbytes = (L.i64 * 6)()
        L.check(lib.tik_pack_block_bytes(C.byref(raw), self.code, first, nbytes))
        names = ("agg", "w_gcn", "b_gcn", "w_tcn", "b_tcn", "w_res_stem")
        dts = (torch.float32, torch.float32 if first else self.tdtype, torch.float32, self.tdtype, torch.float32, torch.float32)
        buf = L.TikPackBuffers()
        for name, dt, nb in zip(names, dts, nbytes):
            if nb == 0:
                continue
            t = torch.empty(nb // dt.itemsize, dtype=dt, device=dev)
            self.keep.append(t)
            self.named[f"b{i}.{name}"] = t
            setattr(buf, name + "_dev", t.data_ptr())
        dbn = backbone.data_bn if isinstance(backbone.data_bn, torch.nn.BatchNorm1d) else None
        with L.on_device(dev):
            L.check(lib.tik_pack_block(C.byref(raw), self.code, first, C.byref(_raw_bn(dbn)) if dbn is not None else None,
                                       C.byref(buf), C.byref(out), L.stream_ptr(dev)))

    def _f32(self, t, name):
        t = t.to(torch.float32).contiguous()
        self.keep.append(t)
        self.named[name] = t
        return t.data_ptr()

    def _act(self, t, name):
        t = t.to(self.tdtype).contiguous()
        self.keep.append(t)
        self.named[name] = t
        return t.data_ptr()


class Plan:
    """One launch plan = kernels + tensor maps over ONE workspace.  A plan belongs to the (device, stream) it was
    made for (Engine keys on both): its workspace is reused by every run, so runs must be stream-ordered."""

    def __init__(self, packed, n_chunk, n_max, T):
        lib = L.lib()
        self.packed = packed
        self.n_chunk, self.n_max, self.T = n_chunk, n_max, T
        nbytes = L.i64(0)
        L.check(lib.tik_stgcn_workspace_bytes(C.byref(packed.net), packed.code, n_chunk, n_max, T, C.byref(nbytes)))
        self.workspace = torch.empty(nbytes.value + 1024, dtype=torch.uint8, device=packed.device)
        base = (self.workspace.data_ptr() + 1023) // 1024 * 1024
        handle = L.vp()
        with L.on_device(packed.device):      # plan_create issues cudaMemcpy / cudaFuncSetAttribute on the current device
            L.check(lib.tik_stgcn_plan_create(C.byref(packed.net), packed.code, n_chunk, n_max, T, C.c_void_p(base),
                                              nbytes.value, C.byref(handle)))
        self.handle = handle
        self.T_out = lib.tik_stgcn_out_frames(C.byref(packed.net), T)
        self.workspace_bytes = nbytes.value
        self._graphs = {}
        self._fin = weakref.finalize(self, lib.tik_stgcn_plan_destroy, handle)

    def launches(self, N):
        return int(L.lib().tik_stgcn_plan_launches(self.handle, N))

    def profile(self, x):
        """One run with CUDA events around every kernel -> {'stem'|'aggregate'|'gemm': (ms, launches)}, gemm flops."""
        p = self.packed
        N = x.shape[0]
        poses = torch.empty((N, self.T_out, max(p.head_out, 1)), dtype=torch.float32, device=x.device)
        ms = (C.c_double * 3)()
        cnt = (L.i64 * 3)()
        fl = C.c_double(0)
        with L.on_device(x):
            L.check(L.lib().tik_stgcn_plan_profile(self.handle, L.ptr(x), N, L.ptr(poses), L.stream_ptr(x.device), ms, cnt,
                                                   C.byref(fl)))
        return {k: (ms[i], int(cnt[i])) for i, k in enumerate(("stem", "aggregate", "gemm"))}, fl.value

    def run_graphed(self, x):
        """Same as run(x)[0] but replays a CUDA graph of the launch sequence (one graph per batch size, at most 4
        kept).  The graph reads a static input buffer (x is copied into it, ~0.2 KB/frame of D2D traffic) and the
        result is copied out of the graph's static output, so callers own what they get."""
        p = self.packed
        N = x.shape[0]
        entry = self._graphs.get(N)
        if entry is None:
            xbuf = torch.empty_like(x)
            poses = torch.empty((N, self.T_out, p.head_out), dtype=torch.float32, device=x.device)

            def enqueue():
                L.check(L.lib().tik_stgcn_plan_run(self.handle, L.ptr(xbuf), N, L.ptr(poses), None, L.stream_ptr(x.device)))
            with L.on_device(x):
                xbuf.copy_(x)
                enqueue()                                             # eager warm-up (function attributes, lazy init)
                torch.cuda.current_stream(x.device).synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    enqueue()
            if len(self._graphs) >= 4:
                self._graphs.pop(next(iter(self._graphs)))
            entry = self._graphs[N] = (graph, poses, xbuf)
        with L.on_device(x):
            entry[2].copy_(x)
            entry[0].replay()
            return entry[1].clone()

    def run_windows(self, seq, n_windows, offset, stride, root):
        """Sliding windows of one resident sequence (F,V,C): window n, frame t = seq[clamp(n*stride + t + offset)],
        root-centred on 0.5*(kp[root[0]] + kp[root[1]]) if root is given.  Nothing is materialised."""
        win, _ = _windowing(seq, offset, stride, root)
        return _launch(self, L.lib().tik_stgcn_plan_run_windows, seq, n_windows, C.byref(win), n_windows)

    def run_seq_windows(self, seq, tables, n_windows, offset, stride, root):
        """run_windows over a ragged batch of sequences packed in seq (frames, V, C): ``tables`` is the int64 device
        tensor (2, n_seqs+1) of frame_start / window_start (inference.sequence_tables).  Window n of sequence s, frame
        t = seq[frame_start[s] + clamp(n*stride + t + offset, 0, F_s - 1)]; windows come out in sequence order."""
        win, seqs = _windowing(seq, offset, stride, root, tables)
        return _launch(self, L.lib().tik_stgcn_plan_run_seq_windows, seq, n_windows, C.byref(win), C.byref(seqs), n_windows)

    def run(self, x, want_feat=False):
        p = self.packed
        N = x.shape[0]
        poses = torch.empty((N, self.T_out, p.head_out), dtype=torch.float32, device=x.device) if p.head_out else None
        feat = torch.empty((N, self.T_out, p.V * p.c_last), dtype=p.tdtype, device=x.device) if want_feat else None
        with L.on_device(x):
            L.check(L.lib().tik_stgcn_plan_run(self.handle, L.ptr(x), N, L.ptr(poses), L.ptr(feat), L.stream_ptr(x.device)))
        return poses, feat


class LatencyPlan:
    """The whole forward for a handful of clips as ONE persistent cooperative kernel (csrc/latency.cu): fp32 arithmetic on
    the fp32 packing, every layer a phase between grid-wide barriers.  Batch-1 windows are launch-bound on the
    throughput plan (19-25 dependent launches); this is one launch."""

    LIMIT_ROWS = 32                     # N * T' head rows

    def __init__(self, packed, n_max, T):
        if packed.code != L.TIK_F32:
            raise ValueError("the latency plan takes the fp32 packing")
        lib = L.lib()
        self.packed, self.n_max, self.T = packed, n_max, T
        nbytes = L.i64(0)
        L.check(lib.tik_stgcn_latency_workspace_bytes(C.byref(packed.net), n_max, T, C.byref(nbytes)))
        self.workspace = torch.empty(nbytes.value + 256, dtype=torch.uint8, device=packed.device)
        base = (self.workspace.data_ptr() + 255) // 256 * 256
        handle = L.vp()
        with L.on_device(packed.device):
            L.check(lib.tik_stgcn_latency_create(C.byref(packed.net), n_max, T, C.c_void_p(base), nbytes.value, C.byref(handle)))
        self.handle = handle
        self.T_out = lib.tik_stgcn_out_frames(C.byref(packed.net), T)
        self.phases = int(lib.tik_stgcn_latency_phases(handle))
        self._fin = weakref.finalize(self, lib.tik_stgcn_latency_destroy, handle)

    def launches(self, N):
        return 1

    def run(self, x):
        return _launch(self, L.lib().tik_stgcn_latency_run, x, x.shape[0], x.shape[0])

    def run_windows(self, seq, n_windows, offset, stride, root):
        win, _ = _windowing(seq, offset, stride, root)
        return _launch(self, L.lib().tik_stgcn_latency_run_windows, seq, n_windows, C.byref(win), n_windows)

    def run_seq_windows(self, seq, tables, n_windows, offset, stride, root):
        """Plan.run_seq_windows in one cooperative launch (n_windows <= n_max)."""
        win, seqs = _windowing(seq, offset, stride, root, tables)
        return _launch(self, L.lib().tik_stgcn_latency_run_seq_windows, seq, n_windows, C.byref(win), C.byref(seqs), n_windows)


def _windowing(seq, offset, stride, root, tables=None):
    """TikWindowing over seq (frames, V, C) and, for a ragged batch, the TikSeqBatch of ``tables`` (2, n_seqs+1) int64
    on seq's device (None without tables)."""
    win = L.TikWindowing(seq.shape[0], offset, stride, root[0] if root else -1, root[1] if root else -1)
    if tables is None:
        return win, None
    if tables.dtype != torch.int64 or tables.dim() != 2 or tables.shape[0] != 2 or not tables.is_contiguous() \
            or tables.device != seq.device:
        raise ValueError("tables must be a contiguous (2, n_seqs+1) int64 tensor on the sequence's device")
    row = tables.stride(0) * tables.element_size()
    return win, L.TikSeqBatch(tables.shape[1] - 1, tables.data_ptr(), tables.data_ptr() + row)


def _launch(plan, entry, x, n, *args):
    """poses (n, T', head_out) fp32 of one run of a Plan or LatencyPlan: entry(handle, x, *args, poses, [feat,] stream),
    where the throughput plan's entry points take a feature output (not requested here) after the poses."""
    poses = torch.empty((n, plan.T_out, plan.packed.head_out), dtype=torch.float32, device=x.device)
    feat = (None,) if isinstance(plan, Plan) else ()
    with L.on_device(x):
        L.check(entry(plan.handle, L.ptr(x), *args, L.ptr(poses), *feat, L.stream_ptr(x.device)))
    return poses


MAX_HEAD_CLIPS = 16384   # clips whose features are kept for one head launch (143 MB in bf16 at T=64)


def default_chunk(T):
    """Clips per backbone pass: up to 256K frames (4096 clips at T=64, ~2.9 GB of bf16 workspace).  Measured on
    B200 (profiles/r1_notes.md): with the current per-layer kernels, launches that fill the machine for longer beat
    L2-sized chunks (128 clips: 23 M frames/s, 1024: 34 M, 4096: 37 M), so chunks are as large as memory allows."""
    return max(1, 262144 // max(T, 1))


class Engine:
    """Per-model cache of packed (BN / bias / edge-importance folded) weights and launch plans.

    Invalidation.  The cache is stamped with every parameter's and buffer's (data_ptr, _version, device) plus the
    scalars that enter the folding (BatchNorm eps, LeakyReLU slope), so optimizer steps, `load_state_dict`, `.to()`
    and any autograd-visible in-place update re-fold automatically.  Writes through ``param.data`` (old-style EMA,
    manual loaders) do NOT bump `_version`; after such a write either call ``invalidate()`` (also exposed as
    ``model.invalidate_packed()`` on the modules), or set ``weight_check = "content"``, which additionally compares a
    strided-sample checksum of every tensor on each call (one small device->host read per forward: safe, but it
    serialises the host with the stream, so it is off by default for the latency path)."""

    def __init__(self, backbone, head_fn=None):
        self._backbone = weakref.ref(backbone)
        self._head_fn = head_fn
        self._packed = {}
        self._plans = {}
        self._stamp = None
        self._watch = None
        self.weight_check = os.environ.get("TIK_WEIGHT_CHECK", "version")

    def invalidate(self):
        """Drop the folded weights and every plan; the next forward re-folds from the module's current tensors."""
        self._packed.clear()
        self._plans.clear()
        self._stamp = None
        self._watch = None

    def _collect(self, backbone, head):
        """The tensors and scalars the folding reads.  Walking the module tree costs ~0.3-0.7 ms of host time, far more
        than a batch-1 forward, so the lists are cached and re-walked only when the cheap stamp below changes (or after
        invalidate() / _apply() / load_state_dict(), which EngineHolder hooks).  Not covered: re-ASSIGNING a Parameter
        or buffer object of an already-run model (`bn.running_mean = t`): call invalidate_packed() after that."""
        extra = [] if head is None else [head[0].weight, head[0].bias, head[2].weight, head[2].bias]
        ts = list(backbone.parameters()) + list(backbone.buffers()) + extra
        bns = [m for m in backbone.modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm)]
        self._watch = (ts, bns)
        return self._watch

    def _tensors(self, backbone, head):
        return (self._watch or self._collect(backbone, head))[0]

    def _stamp_now(self, backbone, head, fresh=False):
        ts, bns = self._collect(backbone, head) if (fresh or self._watch is None) else self._watch
        stamp = (tuple(map(_GET_VERSION, ts)), tuple(map(_GET_PTR, ts)), ts[0].device,
                 tuple(map(_GET_EPS, bns)), None if head is None else float(head[1]))
        if self.weight_check == "content":
            # <= 64 strided samples + the sum of each tensor, reduced on the device, one read-back
            with torch.no_grad():
                sums = torch.stack([t.detach().reshape(-1)[:: max(1, t.numel() // 64)].double().sum() + t.detach().double().sum()
                                    for t in ts if t.numel()])
            stamp += (tuple(sums.tolist()),)
        elif self.weight_check != "version":
            raise ValueError("weight_check must be 'version' or 'content'")
        return stamp

    def _refresh(self, backbone, head):
        """Re-fold if anything the folding reads has changed."""
        stamp = self._stamp_now(backbone, head)
        if stamp != self._stamp:
            stamp = self._stamp_now(backbone, head, fresh=True)      # objects may have been replaced: walk the tree again
            self._packed.clear()
            self._plans.clear()
            self._stamp = stamp

    def plan(self, dtype_name, N, T, chunk=None):
        backbone = self._backbone()
        head = self._head_fn() if self._head_fn else None
        self._refresh(backbone, head)
        if dtype_name not in self._packed:
            self._packed[dtype_name] = PackedNet(backbone, head, dtype_name)
        n_chunk = int(chunk) if chunk else default_chunk(T)
        n_chunk = max(1, min(n_chunk, N))
        n_max = max(n_chunk, min(N, MAX_HEAD_CLIPS))
        dev = self._packed[dtype_name].device
        # a plan's workspace is reused by every run: runs on different streams would race on it, so each stream
        # (and device) gets its own plan
        key = (dtype_name, n_chunk, n_max, T, dev.index, torch.cuda.current_stream(dev).cuda_stream)
        if key not in self._plans:
            if len(self._plans) >= 8:                                    # bound the workspaces kept alive
                self._plans.pop(next(iter(self._plans)))
            self._plans[key] = Plan(self._packed[dtype_name], n_chunk, n_max, T)
        return self._plans[key]


def _latency_plan(self, N, T):
    """Engine.latency_plan: cached LatencyPlan for up to N clips of T frames (fp32 packing, one per device / stream)."""
    backbone = self._backbone()
    head = self._head_fn() if self._head_fn else None
    self._refresh(backbone, head)
    if "fp32" not in self._packed:
        self._packed["fp32"] = PackedNet(backbone, head, "fp32")
    dev = self._packed["fp32"].device
    key = ("latency", int(N), T, dev.index, torch.cuda.current_stream(dev).cuda_stream)
    if key not in self._plans:
        if len(self._plans) >= 8:
            self._plans.pop(next(iter(self._plans)))
        self._plans[key] = LatencyPlan(self._packed["fp32"], int(N), T)
    return self._plans[key]


Engine.latency_plan = _latency_plan


class EngineHolder:
    """Mixin for the modules that own an Engine: the engine (weak reference, ctypes handles, device workspaces) is a
    cache, not state -- it is dropped by pickling / ``torch.save(model)`` / ``copy.deepcopy`` and rebuilt lazily, as
    the reference's plain nn.Modules would allow."""

    _CACHE_ATTRS = ("_engine", "_packed", "_head_state")

    def __getstate__(self):
        state = self.__dict__.copy()
        for k in self._CACHE_ATTRS:
            if k in state:
                state[k] = None
        return state

    def _apply(self, fn, *args, **kwargs):
        # .to() / .cuda() / .float(): buffers are REPLACED by new tensor objects, so the engine's cached lists go stale
        out = super()._apply(fn, *args, **kwargs)
        self.invalidate_packed()
        return out

    def load_state_dict(self, *args, **kwargs):
        out = super().load_state_dict(*args, **kwargs)
        self.invalidate_packed()
        return out

    def invalidate_packed(self):
        """Forget folded weights / plans (call after writing parameters through ``.data`` or re-assigning them)."""
        for m in self.modules():
            if isinstance(m, EngineHolder):
                if getattr(m, "_engine", None) is not None:
                    m._engine.invalidate()
                if "_packed" in m.__dict__:
                    m._packed = None
                if "_head_state" in m.__dict__:
                    m._head_state = None
        return self


def require_cuda_eval(module, x, what):
    if module.training:
        raise NotImplementedError(
            f"{what}: the CUDA path implements eval-mode inference only (BatchNorm is folded); call .eval()")
    if not torch.is_tensor(x):
        raise TypeError(f"{what}: expected a torch.Tensor, got {type(x)}")
    if not x.is_cuda:
        raise RuntimeError(f"{what}: input must be a CUDA tensor -- there is no CPU fallback")
    if x.device.index not in _CHECKED_DEVICES:               # compute capability 10.x, checked once per device
        with L.on_device(x):
            L.check(L.lib().tik_check_device())
        _CHECKED_DEVICES.add(x.device.index)
