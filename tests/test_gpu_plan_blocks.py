"""Each tensor-core kernel of the bf16 network plan (csrc/plan.cu), inside the plan and one block at a time, against
fp64 at its tile edges.

Observing a block.  Networks are built from StgGcn18 layer lists and packed by engine.PackedNet; the plan is created
over a workspace filled with 0xFF bytes (bf16 NaN), so any valid output that depends on memory no kernel wrote (rows
past nv in a partial chunk, frames past T, padding rows) comes out non-finite.  The output of a block that is not the
last one is read through an IDENTITY PROBE block appended behind it (c -> c, stride 1, no residual; after packing,
agg = [I, 0, ...], w_gcn = [I | 0 ...], w_tcn = [0 | I | 0], biases 0): every product in the probe is 1*x or 0*x of a
post-ReLU bf16 value, summed in fp32, so the probe returns its input bit for bit whichever graph-conv kernel runs it.
The plan is deterministic, so the probed output of [b0 .. b_{i-1}] is exactly what block i reads (x_i).  Block i's
graph-convolution output H_i is read from a second network in which block i keeps its gcn / tcn.0 parameters (the
packed gcn tensors are asserted equal) but has stride 1, no residual and an identity temporal conv: every frame of
H_i, stride-2 blocks included.

One rounding stage per comparison.  With x_i and H_i observed,
  * the temporal conv (halo kernel or implicit GEMM) is a TikRowGemm of bf16 operands: rowgemm_reference with the
    existing comparator (R_BF16, C_ACC unchanged);
  * the graph conv is relu(W . bf16(agg(x_i)) + b[node]) (fused kernel: bf16 adjacency, as the plan uploads it;
    aggregate kernel: fp32 adjacency), or relu(agg(bf16(W . x_i)) + b) for 256 input channels.  The rounded
    intermediate is not observable: where its fp64 value lies within the fp32 summation bound of a bf16 rounding
    midpoint, the kernel may round either way, so such an element adds one bf16 ulp of it times the absolute weights
    that carry it to the tolerance; every other element adds nothing;
  * the fused first block: H0 = relu(bf16(Wg) . agg + b1) with the fp64 aggregate of the fp32 in_scale / in_shift /
    agg tables.  The kernel feeds the aggregate as a bf16 hi/lo pair (about 16 bits), so the input term
    sum |w| (2^-16 |agg| + fp32 aggregation bound) is added; then Y0 = rowgemm_reference over the observed H0 plus
    R0 = bf16(Wr') . (s0 x) with the bf16 Wr' that stem_block_prepare derives, under the same input term.
The input terms enter as extra scale, compare(got, ref, S + extra / C_ACC): the comparator itself is unchanged.

Tile cases (gcn_fused_frames, tcn_halo_segment and the stem block's lo = min(T, 13) decide them): see CASES below.
"""
import ctypes as C
import re
import weakref

import numpy as np
import pytest
import torch

from rowgemm_reference import C_ACC, compare, reference, ulp_bf16, verdict

U32 = 2.0 ** -24           # fp32 unit roundoff
HILO = 2.0 ** -16          # relative error of a bf16 hi + lo pair


# ------------------------------------------------------------------------------------------------ fp64 references
def bf16_rn(x):
    """fp64 -> nearest bf16 (ties to even), exactly (no double rounding through fp32), as fp64."""
    u = ulp_bf16(x)
    return torch.round(x / u) * u


def midpoint_slack(a, bound):
    """One bf16 ulp of a where a value within `bound` of a could round to a different bf16 number, else 0."""
    return torch.where(bf16_rn(a - bound) != bf16_rn(a + bound), ulp_bf16(a), torch.zeros_like(a))


def gcn_reference(x, A, w, b, wide):
    """Graph conv of a bf16 block input x (N*V, T, cin) as the kernels round it -> (ref, S, extra), node-major.

    A (K, V, V) adjacency the kernel multiplies, w (cout, K*cin) bf16, b (V, cout).  wide = False: aggregate rounded
    to bf16, then the channel GEMM; wide = True (256 input channels, K = 1): channel GEMM rounded to bf16, then the
    aggregation."""
    K, V = A.shape[0], A.shape[1]
    nv, T, cin = x.shape
    N = nv // V
    xd, Ad, wd, bd = x.double().view(N, V, T, cin), A.double(), w.double(), b.double()
    if wide:
        z = torch.einsum("nvtc,oc->nvto", xd, wd)
        e = C_ACC * torch.einsum("nvtc,oc->nvto", xd.abs(), wd.abs())
        zq, sl = bf16_rn(z), midpoint_slack(z, e)
        ref = torch.einsum("vw,nvto->nwto", Ad[0], zq) + bd[None, :, None, :]
        S = torch.einsum("vw,nvto->nwto", Ad[0].abs(), zq.abs()) + bd.abs()[None, :, None, :]
        extra = torch.einsum("vw,nvto->nwto", Ad[0].abs(), sl)
    else:
        a = torch.einsum("kvw,nvtc->nwtkc", Ad, xd)
        e = max(C_ACC, V * U32) * torch.einsum("kvw,nvtc->nwtkc", Ad.abs(), xd.abs())
        aq, sl = bf16_rn(a).reshape(N, V, T, K * cin), midpoint_slack(a, e).reshape(N, V, T, K * cin)
        ref = aq @ wd.t() + bd[None, :, None, :]
        S = aq.abs() @ wd.abs().t() + bd.abs()[None, :, None, :]
        extra = sl @ wd.abs().t()
    sh = (nv, T, -1)
    return ref.clamp_min(0).reshape(sh), S.reshape(sh), extra.reshape(sh)


def stem_inputs(xw, root, in_scale, in_shift, agg):
    """Block 0's inputs from the raw windows xw (N, T, V, cin) fp32 and the fp32 root (N, T, 1, cin) or None:
    fp64 aggregate (N, T, V, K*cin) of data_bn(x - root), its fp32 evaluation bound, and s0 (x - root)."""
    K, V = agg.shape[0], agg.shape[1]
    N, T, _, cin = xw.shape
    xc = xw.double() - (0 if root is None else root.double())
    s0, o0 = in_scale.double().view(V, cin), in_shift.double().view(V, cin)
    Ad = agg.double()
    a = torch.einsum("kuv,ntuc->ntvkc", Ad, xc * s0 + o0).reshape(N, T, V, K * cin)
    mag = torch.einsum("kuv,ntuc->ntvkc", Ad.abs(), xw.double().abs() * s0.abs() + o0.abs())
    if root is not None:
        mag = mag + root.double().abs()[:, :, :, None, :] * torch.einsum("kuv,uc->vkc", Ad.abs(), s0.abs())
    return a, ((V + 4) * U32 * mag).reshape(N, T, V, K * cin), xc * s0


def stem_h0_reference(a, a_err, wg, b1, hilo):
    """H0 (N*V, T, 64) node-major: relu(wg . a + b1[node]) with the input term of a hi/lo (or fp32) aggregate."""
    N, T, V, _ = a.shape
    wd = wg.double()
    ref = (a @ wd.t() + b1.double()).clamp_min(0)
    S = a.abs() @ wd.abs().t() + b1.double().abs()
    extra = ((HILO if hilo else 0.0) * a.abs() + a_err) @ wd.abs().t()
    nm = lambda t: t.permute(0, 2, 1, 3).reshape(N * V, T, -1)
    return nm(ref), nm(S), nm(extra)


def stem_residual_weights(packed):
    """The bf16 Wr' (64, cin) stem_block_prepare derives from w_res_stem and in_scale (packed_emulator mirrors it)."""
    t = packed.named
    V, cin = packed.V, packed.c_in
    s0 = t["in_scale"].view(V, cin).cpu()
    vb = s0.abs().argmax(dim=0)
    sc = s0[vb, torch.arange(cin)]
    wr = t["b0.w_res_stem"].cpu()[vb, :, torch.arange(cin)].t().double() / sc.double()
    return torch.where(sc[None, :] != 0, wr, torch.zeros_like(wr)).float().bfloat16()


def checked(got, ref, S, extra):
    st = compare(got, ref, S + extra / C_ACC, True)
    return st, verdict(st)


# ------------------------------------------------------------------------------------------------ networks and plans
class Source:
    """Seeded synthetic backbone (PoseRegressor's eight blocks) of one skeleton layout / partition strategy / kt."""

    def __init__(self, layout="coco", strategy="uniform", kt=3, res0=True):
        from oracle import stgcn_port as sp
        from temporal_inverse_kinematics_b200 import synthetic
        self.graph_cfg = dict(layout=layout, strategy=strategy, max_hop=2, dilation=1)
        self.blocks = [(3, 64, 1, res0)] + synthetic.POSE_REGRESSOR_LAYERS[1:]
        self.A = sp.build_adjacency(layout, strategy, 2, 1)
        self.sd = synthetic.make_backbone_state(self.A, self.blocks, kt, seed=5, prefix="")
        self.K, self.V = self.A.shape[0], self.A.shape[1]
        self.kt = kt

    def build(self, spec):
        """spec: [(source block, stride, residual) | ("probe", c)] -> eval CUDA StgGcn18 with the source's parameters."""
        from temporal_inverse_kinematics_b200.st_gcn import StgConfig, StgGcn18, StgLayerConfig
        layers, sd = [], {"A": self.sd["A"]}
        sd.update({k: v for k, v in self.sd.items() if k.startswith("data_bn.")})
        for j, s in enumerate(spec):
            if s[0] == "probe":
                layers.append(StgLayerConfig(s[1], s[1], 1, False))
                continue
            i, stride, res = s
            cin, cout = self.blocks[i][0], self.blocks[i][1]
            layers.append(StgLayerConfig(cin, cout, stride, res))
            for k, v in self.sd.items():
                if k.startswith(f"st_gcn_networks.{i}.") and (res or ".residual." not in k):
                    sd[f"st_gcn_networks.{j}." + k.split(".", 2)[2]] = v
            sd[f"edge_importance.{j}"] = self.sd[f"edge_importance.{i}"]
        m = StgGcn18(StgConfig(layers=layers, temporal_kernel_size=self.kt), self.graph_cfg)
        missing, unexpected = m.load_state_dict(sd, strict=False)
        probes = {j for j, s in enumerate(spec) if s[0] == "probe"}
        assert not unexpected and all(int(re.match(r"\w+\.(\d+)", k).group(1)) in probes for k in missing), missing
        return m.cuda().eval()


def pack(src, spec):
    """PackedNet of spec with every probe made the identity and every "h" block's temporal conv made [0 | I | 0]."""
    from temporal_inverse_kinematics_b200 import engine
    m = src.build([s if s[0] == "probe" else s[:3] for s in spec])
    p = engine.PackedNet(m, None, "bf16")
    t = p.named
    for j, s in enumerate(spec):
        kt = src.kt
        if s[0] == "probe":
            c = s[1]
            eye = torch.eye(c, device="cuda")
            t[f"b{j}.agg"].zero_()[0].copy_(torch.eye(src.V, device="cuda"))
            t[f"b{j}.w_gcn"].zero_()[:, :c].copy_(eye)
            t[f"b{j}.b_gcn"].zero_()
        if s[0] == "probe" or s[-1] == "h":
            c = t[f"b{j}.w_tcn"].shape[0]
            pad = (kt - 1) // 2
            t[f"b{j}.w_tcn"].zero_()[:, pad * c:(pad + 1) * c].copy_(torch.eye(c, device="cuda"))
            t[f"b{j}.b_tcn"].zero_()
    p._model = m
    return p


class Plan:
    """engine.Plan over a workspace of 0xFF bytes; runs return the last block's features node-major."""

    def __init__(self, packed, n_chunk, n_max, T):
        from temporal_inverse_kinematics_b200 import _lib as L
        lib = L.lib()
        self.packed, self.T = packed, T
        nbytes = L.i64(0)
        L.check(lib.tik_stgcn_workspace_bytes(C.byref(packed.net), packed.code, n_chunk, n_max, T, C.byref(nbytes)))
        self.workspace = torch.full((nbytes.value + 1024,), 0xFF, dtype=torch.uint8, device="cuda")
        base = (self.workspace.data_ptr() + 1023) // 1024 * 1024
        handle = L.vp()
        L.check(lib.tik_stgcn_plan_create(C.byref(packed.net), packed.code, n_chunk, n_max, T, C.c_void_p(base),
                                          nbytes.value, C.byref(handle)))
        self.handle = handle
        self.T_out = lib.tik_stgcn_out_frames(C.byref(packed.net), T)
        self._fin = weakref.finalize(self, lib.tik_stgcn_plan_destroy, handle)

    def run(self, inp):
        """inp: ("plain", x (N,T,V,C)) | ("window", seq, n, offset, stride, root) | ("seq", seq, tables, n, offset,
        stride, root) -> (N*V, T', C_last) bf16."""
        from temporal_inverse_kinematics_b200 import _lib as L, engine
        p = self.packed
        kind, x = inp[0], inp[1]
        n = x.shape[0] if kind == "plain" else inp[-4]
        feat = torch.full((n, self.T_out, p.V * p.c_last), float("nan"), dtype=torch.bfloat16, device="cuda")
        lib, s = L.lib(), L.stream_ptr(x.device)
        if kind == "plain":
            L.check(lib.tik_stgcn_plan_run(self.handle, L.ptr(x), n, None, L.ptr(feat), s))
        elif kind == "window":
            win, _ = engine._windowing(x, *inp[3:])
            L.check(lib.tik_stgcn_plan_run_windows(self.handle, L.ptr(x), C.byref(win), n, None, L.ptr(feat), s))
        else:
            win, seqs = engine._windowing(x, *inp[4:], inp[2])
            L.check(lib.tik_stgcn_plan_run_seq_windows(self.handle, L.ptr(x), C.byref(win), C.byref(seqs), n, None,
                                                       L.ptr(feat), s))
        torch.cuda.synchronize()
        return feat.view(n, self.T_out, p.V, p.c_last).permute(0, 2, 1, 3).reshape(n * p.V, self.T_out, p.c_last)


def routes(src):
    """The step names the plan must launch for the source's eight blocks (csrc/plan.cu, its *_supported functions)."""
    names, n = [], len(src.blocks)
    for i, (cin, cout, stride, _) in enumerate(src.blocks):
        res = "conv" if (cin != cout or stride != 1) else "identity"
        if i == 0:
            if src.K == 1 and src.kt == 3 and stride == 1 and src.V <= 17:
                names.append("stem_block")
                continue
            names.append("stem")
        elif src.K == 1 and src.V * 7 <= 128 and (cin, cout) in ((64, 64), (64, 128), (128, 128), (128, 256), (256, 256)):
            names.append("fused_gcn")
        else:
            names += ["aggregate", "gemm"]
        halo = i < n - 1 and res == "identity" and src.kt == 3 and cout in (64, 128)
        names.append("tcn_halo" if halo else "gemm")
    return names


def trace_names(packed, n_chunk, T, x, capfd, monkeypatch):
    """Step names of one Plan.profile run with TIK_PLAN_TRACE set."""
    from temporal_inverse_kinematics_b200 import engine
    monkeypatch.setenv("TIK_PLAN_TRACE", "1")
    plan = Plan(packed, n_chunk, max(n_chunk, x.shape[0]), T)
    capfd.readouterr()
    engine.Plan.profile(plan, x)
    monkeypatch.delenv("TIK_PLAN_TRACE")
    err = capfd.readouterr().err
    return re.findall(r"tik trace: step +\d+ (\w+) +clips=", err)


# ------------------------------------------------------------------------------------------------ inputs
def gather_windows(seq, starts, wstart, T, offset, stride, root):
    """What block 0 reads: window w of sequence s, frame t = seq[starts[s] + clamp(w' stride + t + offset)], and the fp32
    root 0.5 (kp[a] + kp[b]) of each frame (None: no root)."""
    n = wstart[-1]
    out = torch.empty(n, T, seq.shape[1], seq.shape[2])
    for s in range(len(starts) - 1):
        f0, f1 = starts[s], starts[s + 1]
        for w in range(wstart[s], wstart[s + 1]):
            out[w] = seq[((w - wstart[s]) * stride + torch.arange(T) + offset).clamp(0, f1 - f0 - 1) + f0]
    if root is None:
        return out, None
    return out, 0.5 * (out[:, :, root[0]:root[0] + 1] + out[:, :, root[1]:root[1] + 1])


class Case:
    """One network input: `plain` N clips of T frames, `window` n windows of one sequence of F frames, or `seq` a ragged
    batch of sequences; chunk clips per backbone pass (None: all); blocks to check; TIK_HALO_SEG."""

    def __init__(self, name, T, N=2, source=(), mode="plain", chunk=None, blocks=None, halo_seg=None, F=None,
                 lengths=None, offset=0, stride=1, root=None):
        self.name, self.T, self.N, self.source, self.mode, self.chunk = name, T, N, source, mode, chunk
        self.blocks, self.halo_seg = blocks, halo_seg
        self.F, self.lengths, self.offset, self.stride, self.root = F, lengths, offset, stride, root

    def __repr__(self):
        return self.name

    def inputs(self, V):
        """-> (run input for Plan.run, raw windows (N, T, V, 3), root or None) with seeded keypoints."""
        g = torch.Generator().manual_seed(sum(map(ord, self.name)))
        if self.mode == "plain":
            x = torch.randn(self.N, self.T, V, 3, generator=g)
            return ("plain", x.cuda()), x, None
        if self.mode == "window":
            seq = torch.randn(self.F, V, 3, generator=g)
            xw, r = gather_windows(seq, [0, self.F], [0, self.N], self.T, self.offset, self.stride, self.root)
            return ("window", seq.cuda(), self.N, self.offset, self.stride, self.root), xw, r
        from temporal_inverse_kinematics_b200.inference import sequence_tables
        fs, ws = sequence_tables(self.lengths, self.T, self.offset, self.stride)
        seq = torch.randn(int(fs[-1]), V, 3, generator=g)
        xw, r = gather_windows(seq, fs.tolist(), ws.tolist(), self.T, self.offset, self.stride, self.root)
        tables = torch.from_numpy(np.stack([fs, ws])).cuda()
        return ("seq", seq.cuda(), tables, int(ws[-1]), self.offset, self.stride, self.root), xw, r


# Which tile case each T exercises.  Block lengths of the coco network at input length T: b0, b1 at T (64 channels),
# b2 reads T and writes ceil(T/2); b3, b4, b5 at ceil(T/2) (128 channels); b6 at ceil(T/4); b7 at ceil(T/8) (256).
# Fused first block: lo = min(T, 13) output frames per tile, ceil(T / lo) tiles per clip.
# Fused graph conv: gcn_fused_frames balances min(7, 5 at 256 channels)-frame tiles over the block length.
# Halo temporal conv: 64 channels -> at most 190 rows per tile, 128 channels -> 126; whole-clip tile when T + 2 fits
# and no divisor of T scores clearly better, else divisor segments, else a ragged last segment.
CASES = [
    Case("stem_T1", 1, N=3),               # lo = 1: every tap of the stem block reads zero padding; b7 gcn at 1 frame
    Case("stem_T2", 2, N=3),               # lo = 2
    Case("stem_T12", 12),                  # lo = 12, one tile whose last two rows lie past T
    Case("stem_T13", 13),                  # one full 13-frame tile
    Case("stem_T14", 14),                  # 13 + 1; gcn 64 ch at 14 frames = 7 + 7, 128 ch at 7
    Case("stem_T26", 26),                  # two full tiles: an interior tile edge at frame 13
    Case("stem_T27", 27),                  # 13 + 13 + 1
    Case("stem_T40", 40),                  # 13 x 3 + 1; b7 gcn at 5 frames (one 5-frame tile at 256 ch)
    Case("stem_T64", 64),                  # 13 x 4 + 12, the production shape; halo whole clip at 64 (b1) and 32 (b3, b4)
    Case("stem_T65", 65),                  # 13 x 5
    Case("stem_wrap", 64, N=120, blocks=[0]),   # 600 tiles on at most 148 CTAs: both tile buffers cycle twice or more
    Case("stem_res_none", 27, source=(("res0", False),)),   # first block without its residual convolution
    Case("stem_window", 16, N=20, mode="window", F=50, offset=-5, stride=3, root=(11, 12)),   # clamped at both ends
    Case("stem_seq", 13, mode="seq", lengths=[5, 30, 1, 17], offset=-6, root=(11, 12)),      # ragged sequence batch
    Case("gcn_T7", 7),                     # 64 ch: one 7-frame tile; 128 ch at 4
    Case("gcn_T8", 8),                     # 64 ch: 4 + 4 (balanced, not 7 + 1); 128 ch at 4; b7 at 1
    Case("gcn_T15", 15),                   # 64 ch: 5 + 5 + 5; 128 ch at 8 = 4 + 4
    Case("gcn_T16", 16),                   # 64 ch: 6 + 6 + 4 (ceil); 128 ch at 8
    Case("gcn_T28", 28),                   # 128 ch at 14 = 7 + 7
    Case("gcn_T30", 30),                   # 128 ch at 15 = 5 x 3
    Case("gcn_T32", 32),                   # 128 ch at 16; 256 ch (b7) at 4
    Case("gcn_T48", 48),                   # 256 ch at 6 = 3 + 3
    Case("gcn_T88", 88),                   # 256 ch at 11 = 4 + 4 + 3
    Case("halo_T128", 128, N=1),           # 64 ch whole clip at 128 (130 rows); 128 ch at 64 in 32-frame divisor segments
    Case("halo_T254_ragged", 254, N=1),    # 64 ch at 254 = 127 + 127; 128 ch at 127 = 126 + a ragged 1-frame segment
    Case("halo_G_clipped", 8, N=1, chunk=1),    # 19 (64 ch) and 21 (128 ch) row groups fit a tile; nv = 17 clips G
    Case("halo_partial_chunk", 64, N=5, chunk=2),   # chunks of 2, 2, 1 clips: the last tile of a chunk is partial
    Case("halo_seg1", 64, halo_seg=1),     # TIK_HALO_SEG: one-frame segments, every row a halo row
    Case("halo_seg7", 64, halo_seg=7),     # 64 = 9 x 7 + 1, 32 = 4 x 7 + 4: ragged last segments
    Case("halo_seg31", 64, halo_seg=31),   # T - 1 at 128 ch (b3, b4 at 32): 31 + 1; b1: 31 + 31 + 2
    Case("halo_seg63", 64, halo_seg=63),   # T - 1 at 64 ch (b1): 63 + 1 (ignored by b3, b4: longer than their clip)
    Case("openpose", 40, source=(("layout", "openpose"),)),        # V = 18: stem + GEMM first block, fused gcn
    Case("ntu", 20, source=(("layout", "ntu-rgb+d"),)),            # V = 25: stem, aggregate + GEMM
    Case("spatial", 20, source=(("strategy", "spatial"),)),        # K = 3: stem, aggregate + GEMM over 3 partitions
    Case("kt5", 20, source=(("kt", 5),)),                          # five temporal taps: stem, per-tap GEMMs, no halo
]

_SOURCES = {}


def source(key):
    if key not in _SOURCES:
        _SOURCES[key] = Source(**dict(key))
    return _SOURCES[key]


def block_routes(src):
    """Per block: (graph-conv step, temporal-conv step) of routes(); the fused first block is both."""
    flat, out, k = routes(src), [], 0
    for _ in src.blocks:
        if flat[k] == "stem_block":
            out.append(("stem_block", "stem_block"))
            k += 1
            continue
        g = flat[k]
        k += 2 if g == "aggregate" else 1
        out.append((g, flat[k]))
        k += 1
    return out


def _report(case, i, what, st):
    print(f"\n[plan-blocks] case={case.name} block={i} kernel={what} err/tol={st['ratio']:.4f} "
          f"need_c=2^-20*{st['need_c'] * 2 ** 20:.4f} mean_ulp={st['mean_ulp']:+.4f} toward_ulp={st['toward_ulp']:+.4f} "
          f"n_bias={st['n_bias']}")


def check_case(case, capfd, monkeypatch):
    src = source(case.source)
    V = src.V
    inp, xw, root = case.inputs(V)
    N, T = xw.shape[0], case.T
    chunk = case.chunk or N
    if case.halo_seg:
        monkeypatch.setenv("TIK_HALO_SEG", str(case.halo_seg))
    real = [(i, s, r) for i, (_, _, s, r) in enumerate(src.blocks)]
    full = pack(src, real)
    assert trace_names(full, chunk, T, xw.cuda(), capfd, monkeypatch) == routes(src) * -(-N // chunk)   # per chunk
    rts = block_routes(src)
    observed = {}

    def observe(spec):
        key = repr(spec)
        if key not in observed:
            p = pack(src, spec)
            y = Plan(p, chunk, N, T).run(inp)
            observed[key] = (y, p)
        return observed[key]

    last = len(real) - 1
    probe = lambda c: [("probe", c)]
    bad = []
    t = T
    for i in range(len(real)):
        cin, cout, stride, res = src.blocks[i]
        t_out = (t - 1) // stride + 1
        if case.blocks is None or i in case.blocks:
            hspec = real[:i] + [(i, 1, False, "h")] + (probe(cout) if i == 0 else [])
            H, hp = observe(hspec)
            y, yp = observe(real[:i + 1] + probe(cout)) if i < last else observe(real)
            for k in ("agg", "w_gcn", "b_gcn"):
                assert torch.equal(hp.named[f"b{i}.{k}"], yp.named[f"b{i}.{k}"]), k
            assert torch.isfinite(H.float()).all() and torch.isfinite(y.float()).all(), (case.name, i)
            nt = yp.named
            g_route, t_route = rts[i]
            if i == 0:
                a, a_err, xs = stem_inputs(xw.cuda(), None if root is None else root.cuda(), nt["in_scale"],
                                           nt["in_shift"], nt["b0.agg"])
                fused = g_route == "stem_block"
                wg = nt["b0.w_gcn"].bfloat16() if fused else nt["b0.w_gcn"]
                st, v = checked(H, *stem_h0_reference(a, a_err, wg, nt["b0.b_gcn"], fused))
                _report(case, 0, f"{g_route}:H0", st)
                bad += [(i, "H0", v)] if v else []
                if fused:                                   # Y0 = taps over H0 + R0 (bf16 Wr') + b2[node]
                    nvt = lambda q: q.permute(0, 2, 1, 3).reshape(N * V, T, -1)
                    r0 = extra = None
                    if res:
                        wr = stem_residual_weights(yp).cuda().double()
                        r0 = nvt(xs @ wr.t())
                        extra = nvt(xs.abs() @ wr.abs().t()) * (HILO + C_ACC)
                    b2 = nt["b0.b_tcn"].view(-1, cout)
                    ref, S = reference([(H, 1, dt - 1) for dt in range(3)], nt["b0.w_tcn"][:, :3 * cout], b2, N * V, V, T,
                                       act="relu", residual=r0, with_scale=True)
                    st, v = checked(y, ref, S, torch.zeros_like(S) if extra is None else extra)
                    _report(case, 0, "stem_block:Y0", st)
                    bad += [(i, "Y0", v)] if v else []
            else:
                x, _ = observe(real[:i] + probe(cin))
                A = nt[f"b{i}.agg"]
                A = A.bfloat16().float() if g_route == "fused_gcn" else A
                st, v = checked(H, *gcn_reference(x, A, nt[f"b{i}.w_gcn"], nt[f"b{i}.b_gcn"], cin == 256 and g_route == "fused_gcn"))
                _report(case, i, g_route, st)
                bad += [(i, g_route, v)] if v else []
                pad = (src.kt - 1) // 2
                slabs = [(H, stride, dt - pad) for dt in range(src.kt)] + [(x, stride, 0)]   # residual conv or identity slab
                ref, S = reference(slabs, nt[f"b{i}.w_tcn"], nt[f"b{i}.b_tcn"].view(1, -1), N * V, V, t_out, act="relu",
                                   with_scale=True)
                st = compare(y, ref, S, True)
                _report(case, i, t_route, st)
                bad += [(i, t_route, verdict(st))] if verdict(st) else []
        t = t_out
    assert not bad, (case.name, bad)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=repr)
def test_plan_block_matches_fp64(case, capfd, monkeypatch):
    monkeypatch.delenv("TIK_HALO_SEG", raising=False)
    for k in ("TIK_NO_STEM_BLOCK", "TIK_NO_FUSED_GCN", "TIK_NO_TCN_HALO", "TIK_NO_TS"):
        monkeypatch.delenv(k, raising=False)
    check_case(case, capfd, monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("c", [64, 128, 256])
@pytest.mark.parametrize("strategy", ["uniform", "spatial"])
def test_identity_probe_is_exact(c, strategy, capfd, monkeypatch):
    """[net, probe] and [net, probe, probe] give the same bits, with the probe's graph conv on the fused kernel (K = 1)
    and on aggregate + GEMM (K = 3), at 64, 128 and 256 channels."""
    src = source((("strategy", strategy),))
    prefix = [(i, s, r) for i, (_, co, s, r) in enumerate(src.blocks)][:{64: 2, 128: 5, 256: 7}[c]]
    case = Case("probe", 20, N=3)
    inp, xw, _ = case.inputs(src.V)
    p1, p2 = pack(src, prefix + [("probe", c)]), pack(src, prefix + [("probe", c), ("probe", c)])
    names = trace_names(p2, 3, 20, xw.cuda(), capfd, monkeypatch)
    gcn = "fused_gcn" if strategy == "uniform" else "aggregate"
    assert names[-4:] == [gcn, "gemm"] * 2 if gcn == "fused_gcn" else names[-6:] == [gcn, "gemm", "gemm"] * 2, names
    y1, y2 = Plan(p1, 3, 3, 20).run(inp), Plan(p2, 3, 3, 20).run(inp)
    assert torch.isfinite(y1.float()).all() and bool((y1 > 0).any())
    assert torch.equal(y1, y2)


# ------------------------------------------------------------------------------------------------ CPU: the bounds
# Each bound accepts an fp32-accumulation, round-to-nearest emulation of its kernel and rejects the mistakes such a
# kernel could make.  V = 17 nodes, a sparse random adjacency, post-ReLU bf16 activations.
def _operands(seed, n=2, t=27, cin=64, cout=64, K=1, V=17):
    g = torch.Generator().manual_seed(seed)
    A = torch.rand(K, V, V, generator=g) * (torch.rand(K, V, V, generator=g) > 0.7)
    x = torch.relu(torch.randn(n * V, t, cin, generator=g)).bfloat16()
    w = (torch.randn(cout, K * cin, generator=g) / (K * cin) ** 0.5).bfloat16()
    b = torch.randn(V, cout, generator=g) * 0.1
    return A, x, w, b


def _gcn_kernel(x, A, w, b, wide, round_intermediate=True, bias_shift=0):
    """The graph-conv kernels' arithmetic in fp32 with RN conversions (fused / aggregate + GEMM, or the wide order)."""
    K, V = A.shape[0], A.shape[1]
    nv, T, cin = x.shape
    xf = x.float().view(nv // V, V, T, cin)
    b = b.roll(bias_shift, 0)
    if wide:
        z = xf @ w.float().t()
        z = z.bfloat16().float() if round_intermediate else z
        y = torch.einsum("vw,nvto->nwto", A[0], z) + b[None, :, None, :]
    else:
        a = torch.einsum("kvw,nvtc->nwtkc", A, xf).reshape(nv // V, V, T, K * cin)
        a = a.bfloat16().float() if round_intermediate else a
        y = a @ w.float().t() + b[None, :, None, :]
    return torch.relu(y).bfloat16().reshape(nv, T, -1)


GCN_SHAPES = {"fused_k1": dict(K=1, wide=False), "aggregate_k3": dict(K=3, wide=False),
              "wide_256": dict(K=1, cin=256, cout=256, t=8, wide=True)}


@pytest.mark.parametrize("shape", sorted(GCN_SHAPES))
def test_gcn_bound_accepts_fp32_rn_emulation(shape):
    kw = dict(GCN_SHAPES[shape])
    wide = kw.pop("wide")
    A, x, w, b = _operands(7, **kw)
    st, bad = checked(_gcn_kernel(x, A, w, b, wide), *gcn_reference(x, A, w, b, wide))
    assert bad == [] and st["n_bias"] >= 4096, st


@pytest.mark.parametrize("shape,mistake", [(s, m) for s in sorted(GCN_SHAPES) for m in ("bias_of_next_node", "unrounded")])
def test_gcn_bound_rejects_kernel_mistakes(shape, mistake):
    """The neighbouring node's bias; the intermediate (aggregate, or the wide kernel's channel GEMM) not rounded."""
    kw = dict(GCN_SHAPES[shape])
    wide = kw.pop("wide")
    A, x, w, b = _operands(7, **kw)
    got = _gcn_kernel(x, A, w, b, wide, round_intermediate=mistake != "unrounded",
                      bias_shift=1 if mistake == "bias_of_next_node" else 0)
    assert checked(got, *gcn_reference(x, A, w, b, wide))[1] != []


def _stem_operands(seed=3, n=2, T=27, V=17):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, T, V, 3, generator=g)
    s0, o0 = 0.6 + 0.8 * torch.rand(V * 3, generator=g), 0.1 * torch.randn(V * 3, generator=g)
    A = torch.rand(1, V, V, generator=g) * (torch.rand(1, V, V, generator=g) > 0.7) + 0.5 * torch.eye(V)
    wg = torch.randn(64, 3, generator=g)
    b1 = 0.1 * torch.randn(V, 64, generator=g)
    wt = (torch.randn(64, 192, generator=g) / 192 ** 0.5).bfloat16()
    b2 = 0.1 * torch.randn(V, 64, generator=g)
    wr = torch.randn(64, 3, generator=g).bfloat16()
    return dict(x=x, s0=s0, o0=o0, A=A, wg=wg, b1=b1, wt=wt, b2=b2, wr=wr)


def _hilo(a, lo=True):
    hi = a.bfloat16().float()
    return hi + (a - hi).bfloat16().float() if lo else hi


def _stem_kernel_h0(o, lo=True):
    """The stem block's H0 in fp32: aggregate, hi/lo split, bf16 weights, + b1, ReLU, bf16; node-major."""
    n, T, V, _ = o["x"].shape
    agg = torch.einsum("kuv,ntuc->ntvc", o["A"], o["x"] * o["s0"].view(V, 3) + o["o0"].view(V, 3))
    h = torch.relu(_hilo(agg, lo) @ o["wg"].bfloat16().float().t() + o["b1"]).bfloat16()
    return h.permute(0, 2, 1, 3).reshape(n * V, T, 64)


def _cut_gather(L):
    """gather() of a kernel that zero-fills instead of reading across a boundary every L frames (stride 1)."""
    def g(a, t_out, t_mul, t_off):
        from rowgemm_reference import gather
        rows = gather(a, t_out, t_mul, t_off)
        ts = torch.arange(t_out)
        rows[:, (ts + t_off) // L != ts // L] = 0
        return rows
    return g


def _stem_y0(o, h0, gather_fn=None, pad_relu_b1=False):
    """-> (fp64 Y0, S, extra) over the bf16 H0 and R0 = Wr' . (s0 x), as the bound sees it, and a kernel-order result."""
    from rowgemm_reference import gather
    n, T, V, _ = o["x"].shape
    xs = o["x"].double() * o["s0"].double().view(V, 3)
    nvt = lambda q: q.permute(0, 2, 1, 3).reshape(n * V, T, -1)
    r0 = nvt(xs @ o["wr"].double().t())
    extra = nvt(xs.abs() @ o["wr"].double().abs().t()) * (HILO + C_ACC)
    ref, S = reference([(h0, 1, dt - 1) for dt in range(3)], o["wt"], o["b2"], n * V, V, T, act="relu", residual=r0,
                       with_scale=True)
    g = gather_fn or gather
    hk = h0
    if pad_relu_b1:                                   # clip-end padding rows hold relu(b1[node]) instead of zero
        edge = torch.relu(o["b1"]).bfloat16().repeat(n, 1)[:, None, :]
        hk = torch.cat([edge, h0, edge], dim=1)
    taps = sum(g(hk, T, 1, dt - 1 + (1 if pad_relu_b1 else 0)).float() @ o["wt"][:, 64 * dt:64 * dt + 64].float().t()
               for dt in range(3))
    r0k = nvt(_hilo((o["x"] * o["s0"].view(V, 3)).float()) @ o["wr"].float().t())
    got = torch.relu(taps + r0k + o["b2"].repeat(n, 1)[:, None, :]).bfloat16()
    return got, ref, S, extra


def test_stem_bounds_accept_fp32_rn_emulation():
    o = _stem_operands()
    n, T, V, _ = o["x"].shape
    a, a_err, _ = stem_inputs(o["x"], None, o["s0"], o["o0"], o["A"])
    h0 = _stem_kernel_h0(o)
    st, bad = checked(h0, *stem_h0_reference(a, a_err, o["wg"].bfloat16(), o["b1"], True))
    assert bad == [] and st["n_bias"] >= 4096, st
    st, bad = checked(*_stem_y0(o, h0))
    assert bad == [] and st["n_bias"] >= 4096, st


@pytest.mark.parametrize("mistake", ["lo_half_dropped", "padding_relu_b1", "tap_across_13_frame_tile_edge"])
def test_stem_bounds_reject_kernel_mistakes(mistake):
    o = _stem_operands()
    h0 = _stem_kernel_h0(o)
    if mistake == "lo_half_dropped":
        a, a_err, _ = stem_inputs(o["x"], None, o["s0"], o["o0"], o["A"])
        bad = checked(_stem_kernel_h0(o, lo=False), *stem_h0_reference(a, a_err, o["wg"].bfloat16(), o["b1"], True))[1]
    else:
        bad = checked(*_stem_y0(o, h0, gather_fn=_cut_gather(13) if mistake.startswith("tap") else None,
                                pad_relu_b1=mistake == "padding_relu_b1"))[1]
    assert bad != [], mistake


def _halo_case(L=10, T=27):
    """A stride-1 64-channel temporal conv with the identity slab, cut into segments of L frames (last one ragged)."""
    A, x, w, b = _operands(11, t=T)
    g = torch.Generator().manual_seed(12)
    h = torch.relu(torch.randn(x.shape, generator=g)).bfloat16()
    wt = torch.cat([(torch.randn(64, 192, generator=g) / 192 ** 0.5), torch.eye(64)], dim=1).bfloat16()
    bt = 0.1 * torch.randn(1, 64, generator=g)
    slabs = [(h, 1, -1), (h, 1, 0), (h, 1, 1), (x, 1, 0)]
    return slabs, wt, bt, x.shape[0], 17, T, L


def _halo_run(slabs, wt, bt, nv, V, T, gather_fn=None):
    from rowgemm_reference import gather
    return reference(slabs, wt, bt, nv, V, T, act="relu", gather_fn=gather_fn or gather).float().bfloat16()


def test_halo_bound_accepts_fp32_rn_emulation():
    import packed_emulator
    slabs, wt, bt, nv, V, T, L = _halo_case()
    got = packed_emulator.rowgemm(slabs, wt, bt, V, T, "relu", quant=torch.bfloat16)
    ref, S = reference(slabs, wt, bt, nv, V, T, act="relu", with_scale=True)
    st = compare(got, ref, S, True)
    assert verdict(st) == [] and st["n_bias"] >= 4096, st


@pytest.mark.parametrize("mistake", ["zero_halo_at_interior_segment", "stale_row_in_ragged_segment",
                                     "residual_of_other_row_group"])
def test_halo_bound_rejects_kernel_mistakes(mistake):
    slabs, wt, bt, nv, V, T, L = _halo_case()
    ref, S = reference(slabs, wt, bt, nv, V, T, act="relu", with_scale=True)
    if mistake == "zero_halo_at_interior_segment":
        got = _halo_run(slabs, wt, bt, nv, V, T, gather_fn=_cut_gather(L))
    elif mistake == "stale_row_in_ragged_segment":
        got = _halo_run(slabs, wt, bt, nv, V, T)
        last = (T - 1) // L * L
        got[:, last:] = got.roll(1, 0)[:, last:]
    else:
        x = slabs[3][0]
        got = _halo_run(slabs[:3] + [(x.roll(1, 0), 1, 0)], wt, bt, nv, V, T)
    assert verdict(compare(got, ref, S, True)) != [], mistake
