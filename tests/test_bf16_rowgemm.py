"""tik_rowgemm in bf16 (csrc/stgcn_umma.cu: rowgemm_umma_kernel<BN, ACT> and the weight-stationary rowgemm_ts_kernel)
against an fp64 evaluation of the TikRowGemm definition, at every launch configuration umma_prepare can select.

Error model.  The operands are bf16, so they and every product a_k*w_k are exact in fp64 (and in fp32).  The kernel
sums all of K in one fp32 accumulator in tensor memory, adds the fp32 bias and the bf16 residual in fp32, applies the
activation in fp32, and rounds the result to bf16 with RN ('node' / 'time' layouts) or stores it as fp32 ('rows_f32').
Per element, with S = sum_k |a_k w_k| + |bias| + |residual| computed in fp64 beside the reference:

    |got - ref| <= r |ref| + c S        r = 2^-8 for bf16 outputs (half an ulp), 0 for rows_f32

c bounds the fp32 accumulation error relative to S.  Over the whole case matrix below (random-sign data, K from 64
to 4544) the smallest c that passes every element was 0.091 * 2^-18 = 2^-21.5 on an NVIDIA B200 (1,000 W power
limit), at the iterative head's fc2 (K = 512); C_ACC = 2^-20 leaves a factor of 2.7 over it.

A per-element bound of half an ulp cannot see an output conversion that rounds in one direction.  So over the
well-conditioned elements of every large bf16 case (where c S is at most 1/16 ulp) the mean of (got - ref) / ulp and
of sign(ref) (got - ref) / ulp must both stay below 0.1 ulp: RN gives about 0 (at most 0.0031 measured), RZ -0.5,
RU / RD +-0.5.

The CPU tests at the top show that this comparator accepts an fp32 accumulation rounded to nearest and rejects the
plausible kernel mistakes (a dropped K chunk, a tap read one frame off, padding at the wrong clip end, the neighbouring
node's bias or row's residual, a missed row group, the wrong LeakyReLU slope, truncating output conversion).
"""
import ctypes as C

import pytest
import torch

from rowgemm_reference import BIAS_MIN_ELEMS, compare, gather, reference, to_layout, ulp_bf16, verdict

ACT_CODE = {"none": 0, "relu": 1, "leaky": 2}
TUNING_VARS = ("TIK_UMMA_GROUP", "TIK_UMMA_OPT", "TIK_UMMA_BN", "TIK_NO_TS", "TIK_NO_ROWGEMM_CACHE")


# ------------------------------------------------------------------------------------------------ cases
class Case:
    """One tik_rowgemm call: n clips of v nodes (nv = n*v row groups), slabs [(c, t_mul, t_off, t_in)]; `kern` is the
    kernel umma_prepare must pick with no tuning variable set: 'ts' or the SS kernel's BN."""

    def __init__(self, name, family, kern, n=2, v=17, t_out=16, slabs=None, c_out=64, act="relu", slope=0.01,
                 per_node=False, res=False, layout="node", c_valid=None):
        self.name, self.family, self.kern = name, family, kern
        self.n, self.v, self.nv, self.t_out = n, v, n * v, t_out
        self.slabs = slabs if slabs is not None else [(64, 1, o, t_out) for o in (-1, 0, 1)]
        self.c_out, self.act, self.slope = c_out, act, float(torch.tensor(slope, dtype=torch.float32))
        self.per_node, self.res, self.layout = per_node, res, layout
        self.c_valid = c_valid
        self.ktot = sum(s[0] for s in self.slabs)
        self.bf16_out = layout != "rows_f32"

    def __repr__(self):
        return self.name

    def inputs(self, seed=0):
        """Seeded CPU tensors: bf16 activations / weights / residual, fp32 bias."""
        g = torch.Generator().manual_seed(seed)
        slabs = [((torch.randn(self.nv, t_in, c, generator=g)).bfloat16(), m, o) for c, m, o, t_in in self.slabs]
        w = (torch.randn(self.c_out, self.ktot, generator=g) / self.ktot ** 0.5).bfloat16()
        bias = torch.randn(self.v if self.per_node else 1, self.c_out, generator=g)
        res = torch.randn(self.nv, self.t_out, self.c_out, generator=g).bfloat16() if self.res else None
        return {"slabs": slabs, "w": w, "bias": bias, "res": res}

    def reference(self, inp, with_scale=True, **kw):
        args = dict(act=self.act, slope=self.slope, residual=inp["res"], out_layout=self.layout, c_out_valid=self.c_valid,
                    with_scale=with_scale)
        args.update(kw)
        return reference(inp["slabs"], inp["w"], inp["bias"], self.nv, self.v, self.t_out, **args)

    def out_shape(self):
        if self.layout == "node":
            return (self.nv, self.t_out, self.c_out)
        if self.layout == "time":
            return (self.n, self.t_out, self.v, self.c_out)
        return (self.nv * self.t_out, self.c_valid or self.c_out)


def _taps(c, t_mul, t_in, offs=(-1, 0, 1)):
    return [(c, t_mul, o, t_in) for o in offs]


# ------------------------------------------------------------------------------------------------ CPU: the comparator
def _round_like_kernel(x, bf16_out, mode="rn"):
    """fp64 result -> what the epilogue stores: fp32, then bf16 with RN (or RZ: the low 16 bits dropped)."""
    x32 = x.float()
    if not bf16_out:
        return x32.double()
    if mode == "rn":
        return x32.bfloat16().double()
    return (x32.view(torch.int32) & -65536).view(torch.float32).double()


def _fp32_kernel_order(case, inp):
    """The kernel's arithmetic in fp32: one accumulator over 64-column K chunks, + bias, + residual, activation."""
    acc = torch.zeros(case.nv, case.t_out, case.c_out, dtype=torch.float32)
    koff = 0
    w = inp["w"].float()
    for a, m, o in inp["slabs"]:
        rows = gather(a, case.t_out, m, o).float()
        for c0 in range(0, a.shape[2], 64):
            acc += rows[..., c0:c0 + 64] @ w[:, koff + c0:koff + c0 + 64].t()
        koff += a.shape[2]
    b = inp["bias"]
    acc += b[torch.arange(case.nv) % case.v][:, None, :] if b.shape[0] > 1 else b[0]
    if inp["res"] is not None:
        acc += inp["res"].float()
    if case.act == "relu":
        acc = acc.clamp_min(0)
    elif case.act == "leaky":
        acc = torch.where(acc > 0, acc, acc * case.slope)
    y = to_layout(acc, case.nv, case.v, case.t_out, case.layout, case.c_valid)
    return y.bfloat16().double() if case.bf16_out else y.double()


MUT_CASES = {
    # three stride-1 taps, per-node bias (V = 5), identity residual, LeakyReLU 0.2, node-major bf16
    "taps_res_leaky": Case("taps_res_leaky", "cpu", None, n=2, v=5, t_out=12, slabs=_taps(64, 1, 12), c_out=64,
                           act="leaky", slope=0.2, per_node=True, res=True),
    # stride-2 taps + a t_mul = 1 residual slab, ReLU, time-major bf16
    "stride2_mixed_time": Case("stride2_mixed_time", "cpu", None, n=3, v=17, t_out=8,
                               slabs=_taps(64, 2, 16) + [(64, 1, 0, 8)], c_out=128, layout="time"),
    # head-like: 300 rows, LeakyReLU 0.2, fp32 rows with 66 of 128 columns stored
    "head_rows_f32": Case("head_rows_f32", "cpu", None, n=1, v=1, t_out=300, slabs=[(128, 1, 0, 300), (128, 1, 0, 300)],
                          c_out=128, act="leaky", slope=0.2, layout="rows_f32", c_valid=66),
}


def _wrong_edge_gather(a, t_out, t_mul, t_off):
    """Zero padding at the wrong clip end: the rows that should be zero read the clamped frame instead, and as many
    rows at the other end are zeroed."""
    nv, t_in, c = a.shape
    ts = torch.arange(t_out) * t_mul + t_off
    ok = ((ts >= 0) & (ts < t_in)).flip(0)
    rows = torch.zeros(nv, t_out, c, dtype=torch.float64)
    rows[:, ok] = a.double()[:, ts.clamp(0, t_in - 1)[ok]]
    return rows


def _shift_tap(inp, d):
    a, m, o = inp["slabs"][0]
    return dict(inp, slabs=[(a, m, o + d)] + inp["slabs"][1:])


def _missed_last_group(case, inp):
    y = case.reference(inp, with_scale=False, out_layout="node")
    if case.nv > 1:
        y[-1] = 0
    else:
        y[:, -(case.t_out % 128 or 128):] = 0          # the last tile of rows
    return to_layout(y, case.nv, case.v, case.t_out, case.layout, case.c_valid)


def _drop_last_chunk(case, inp):
    w = inp["w"].clone()
    w[:, -64:] = 0
    return case.reference(dict(inp, w=w), with_scale=False)


def _neighbour_residual(case, inp):
    res = inp["res"].reshape(-1, case.c_out).roll(1, 0).reshape(inp["res"].shape)
    return case.reference(dict(inp, res=res), with_scale=False)


MUTATIONS = {
    "drop_last_k_chunk": _drop_last_chunk,
    "tap_one_frame_early": lambda case, inp: case.reference(_shift_tap(inp, -1), with_scale=False),
    "tap_one_frame_late": lambda case, inp: case.reference(_shift_tap(inp, +1), with_scale=False),
    "padding_at_wrong_edge": lambda case, inp: case.reference(inp, with_scale=False, gather_fn=_wrong_edge_gather),
    "bias_of_next_node": lambda case, inp: case.reference(dict(inp, bias=inp["bias"].roll(-1, 0)), with_scale=False),
    "residual_of_neighbour_row": _neighbour_residual,
    "missed_last_row_group": _missed_last_group,
    "leaky_slope_0.01_for_0.2": lambda case, inp: case.reference(inp, with_scale=False, slope=0.01),
    "rz_output_rounding": None,                       # the exact result, rounded toward zero
}

def _pads(case):
    """Does any slab read a frame outside [0, t_in)?"""
    return any(o < 0 or (case.t_out - 1) * m + o >= t_in for _, m, o, t_in in case.slabs)


MUTATION_CASES = [(c, m) for c in MUT_CASES for m in MUTATIONS
                  if not (m == "bias_of_next_node" and not MUT_CASES[c].per_node)
                  and not (m == "residual_of_neighbour_row" and not MUT_CASES[c].res)
                  and not (m == "leaky_slope_0.01_for_0.2" and MUT_CASES[c].act != "leaky")
                  and not (m == "rz_output_rounding" and not MUT_CASES[c].bf16_out)
                  and not (m == "padding_at_wrong_edge" and not _pads(MUT_CASES[c]))]


@pytest.mark.parametrize("name", sorted(MUT_CASES))
def test_comparator_accepts_fp32_accumulation_rounded_to_nearest(name):
    case = MUT_CASES[name]
    inp = case.inputs(seed=3)
    ref, scale = case.reference(inp)
    assert verdict(compare(_round_like_kernel(ref, case.bf16_out), ref, scale, case.bf16_out)) == []
    st = compare(_fp32_kernel_order(case, inp), ref, scale, case.bf16_out)
    assert verdict(st) == [], st
    if case.bf16_out:
        assert st["n_bias"] >= BIAS_MIN_ELEMS, st      # the bias check is active on this case


@pytest.mark.parametrize("name,mutation", MUTATION_CASES)
def test_comparator_rejects_kernel_mistakes(name, mutation):
    case = MUT_CASES[name]
    inp = case.inputs(seed=3)
    ref, scale = case.reference(inp)
    if MUTATIONS[mutation] is None:
        got = _round_like_kernel(ref, case.bf16_out, mode="rz")
    else:
        got = _round_like_kernel(MUTATIONS[mutation](case, inp), case.bf16_out)
    assert verdict(compare(got, ref, scale, case.bf16_out)) != [], mutation


def test_ulp_bf16():
    x = torch.tensor([1.0, 1.5, -3.0, 2.0 ** -20, 255.0, 256.0], dtype=torch.float64)
    assert ulp_bf16(x).tolist() == [2.0 ** -7, 2.0 ** -7, 2.0 ** -6, 2.0 ** -27, 1.0, 2.0]


def test_empty_rowgemm_is_a_no_op_for_both_dtypes():
    """nv = 0 through the C ABI with non-null (never dereferenced) pointers: fp32 and bf16 both return TIK_OK without
    preparing or launching anything, so no device is needed."""
    from temporal_inverse_kinematics_b200 import _lib as L
    g = L.TikRowGemm()
    g.n_slabs = 1
    g.slabs[0].a_dev, g.slabs[0].c, g.slabs[0].t_in, g.slabs[0].t_mul, g.slabs[0].t_off = 0x10000, 64, 4, 1, 0
    g.w_dev, g.bias_dev, g.out_dev = 0x20000, 0x30000, 0x40000
    g.nv, g.v, g.t_out, g.c_out, g.c_out_valid = 0, 17, 4, 64, 64
    g.act, g.res_kind, g.out_layout = L.ACT_RELU, L.RES_NONE, L.OUT_NODE_MAJOR
    for dtype in (L.TIK_F32, L.TIK_BF16):
        assert L.lib().tik_rowgemm(dtype, C.byref(g), None) == 0, L.lib().tik_last_error()


# ------------------------------------------------------------------------------------------------ GPU: the case matrix
def _case_matrix():
    cs = []
    # N tile width from c_out: BN = 256 | 128 | 64, several N tiles at 192, 320, 384, 512
    for c_out, kern in [(64, "ts"), (128, "ts"), (192, 64), (256, 256), (320, 64), (384, 128), (512, 256)]:
        cs.append(Case(f"bn_c{c_out}", "bn", kern, c_out=c_out, slabs=_taps(64 if c_out != 128 else 128, 1, 16)))
    # TS eligibility at its K limit: 512 is weight-stationary, 576 is not
    cs.append(Case("ktot512", "ts_vs_ss", "ts", c_out=128, slabs=_taps(128, 1, 16) + [(128, 1, 0, 16)]))
    cs.append(Case("ktot576", "ts_vs_ss", 128, c_out=128, slabs=_taps(128, 1, 16) + [(128, 1, 0, 16), (64, 1, 0, 16)]))
    # epilogue stores without TMA: time-major and fp32 rows with c_out_valid < c_out
    cs.append(Case("time_c256", "epilogue", 256, n=3, t_out=4, slabs=_taps(256, 2, 8), c_out=256, layout="time"))
    cs.append(Case("time_c64", "epilogue", 64, n=3, t_out=9, slabs=_taps(64, 1, 9), c_out=64, act="none", layout="time"))
    cs.append(Case("rows_f32_66_of_128", "epilogue", 128, n=1, v=1, t_out=300, slabs=[(512, 1, 0, 300)], c_out=128,
                   act="none", layout="rows_f32", c_valid=66))
    cs.append(Case("rows_f32_132_of_192", "epilogue", 64, n=1, v=1, t_out=300, slabs=[(512, 1, 0, 300)], c_out=192,
                   act="none", layout="rows_f32", c_valid=132))
    # tile geometry: tt = min(t_out, 128), vv = 128 / tt -> dead rows, ragged row groups, several frame tiles;
    # nv = 7 is below vv up to t_out = 9 and not a multiple of vv above it.  TS and SS alternate.
    for i, t in enumerate([1, 2, 5, 9, 63, 64, 65, 127, 128, 129, 200, 300]):
        if i % 2 == 0:
            cs.append(Case(f"t_out{t}_ts", "geometry", "ts", n=1, v=7, t_out=t, slabs=_taps(64, 1, t), c_out=128))
        else:
            cs.append(Case(f"t_out{t}_ss", "geometry", 64, n=1, v=7, t_out=t, slabs=_taps(64, 1, t), c_out=64,
                           per_node=True))
    cs.append(Case("t_mul2", "geometry", "ts", n=1, v=7, t_out=64, slabs=_taps(64, 2, 128), c_out=128))
    cs.append(Case("t_mul3_ts", "geometry", "ts", n=1, v=7, t_out=100, slabs=_taps(64, 3, 300), c_out=128))      # tt 85
    cs.append(Case("t_mul3_ss", "geometry", 64, n=1, v=7, t_out=100, slabs=_taps(64, 3, 300), c_out=64, per_node=True))
    cs.append(Case("t_mul8_ts", "geometry", "ts", n=1, v=7, t_out=40, slabs=_taps(64, 8, 320), c_out=128))       # tt 32
    cs.append(Case("t_mul8_ss", "geometry", 64, n=1, v=7, t_out=40, slabs=_taps(64, 8, 320), c_out=64, per_node=True))
    cs.append(Case("t_off_pm2_ts", "geometry", "ts", n=2, v=5, t_out=11, slabs=_taps(64, 1, 11, range(-2, 3)), c_out=128))
    cs.append(Case("t_off_pm2_ss", "geometry", 64, n=2, v=5, t_out=11, slabs=_taps(64, 1, 11, range(-2, 3)), c_out=64,
                   per_node=True))
    cs.append(Case("t_in_short", "geometry", "ts", n=1, v=7, t_out=20, slabs=_taps(64, 2, 35), c_out=128))
    cs.append(Case("t_in_long", "geometry", 64, n=1, v=7, t_out=20, slabs=_taps(64, 2, 45), c_out=64, per_node=True))
    cs.append(Case("nv1_ts", "geometry", "ts", n=1, v=1, t_out=5, slabs=_taps(64, 1, 5), c_out=64))
    cs.append(Case("nv1_ss", "geometry", 128, n=1, v=1, t_out=130, slabs=_taps(64, 1, 130), c_out=128, res=True))
    # mixed slabs: stride-2 taps + the t_mul = 1 residual slab the plan builds for res_as_slab
    cs.append(Case("mixed_slabs_ts", "mixed", "ts", n=2, t_out=16, slabs=_taps(128, 2, 32) + [(128, 1, 0, 16)], c_out=128))
    cs.append(Case("mixed_slabs_ss", "mixed", 256, n=2, t_out=16, slabs=_taps(128, 2, 32) + [(128, 1, 0, 16)], c_out=256))
    # bias tables and the identity residual
    for v, c_out, kern in [(17, 64, 64), (18, 128, 128), (25, 256, 256), (32, 128, 128)]:
        cs.append(Case(f"bias_v{v}", "bias_res", kern, n=3, v=v, c_out=c_out, per_node=True))
    cs.append(Case("bias_v1", "bias_res", "ts", n=5, v=1, c_out=128))
    cs.append(Case("bias_shared_ss", "bias_res", 64, n=3, c_out=320))
    for c_out in (64, 128, 256):
        cs.append(Case(f"residual_c{c_out}", "bias_res", c_out, n=2, c_out=c_out, res=True))
    cs.append(Case("residual_time", "bias_res", 128, n=2, c_out=128, res=True, per_node=True, layout="time"))
    # activations on each kernel and on fp32 rows
    for act, slope in [("none", 0.01), ("relu", 0.01), ("leaky", 0.01), ("leaky", 0.2)]:
        tag = act if act != "leaky" else f"leaky{slope}"
        cs.append(Case(f"act_{tag}_ts", "act", "ts", c_out=128, act=act, slope=slope))
        cs.append(Case(f"act_{tag}_ss", "act", 128, c_out=128, act=act, slope=slope, per_node=True))
        cs.append(Case(f"act_{tag}_rows_f32", "act", 128, n=1, v=1, t_out=200, slabs=[(256, 1, 0, 200)], c_out=128,
                       act=act, slope=slope, layout="rows_f32", c_valid=100))
    # persistent loop: 1088 tiles (each CTA cycles both accumulators and staging tiles ~7 times), and 9 tiles
    cs.append(Case("tiles1088_ss", "persistent", 64, n=64, t_out=128, slabs=[(64, 1, 0, 128)], c_out=64, per_node=True))
    cs.append(Case("tiles1088_ts", "persistent", "ts", n=64, t_out=128, slabs=[(64, 1, 0, 128)], c_out=128))
    cs.append(Case("tiles9", "persistent", 64, n=1, t_out=64, slabs=_taps(64, 1, 64), c_out=64, per_node=True))
    # production shapes: the plan's head, the iterative head's three layers, the b2 / b5 / b6 temporal convolutions
    cs.append(Case("head1", "production", 256, n=1, v=1, t_out=16384, slabs=[(4352, 1, 0, 16384)], c_out=512, act="leaky"))
    cs.append(Case("head2", "production", 128, n=1, v=1, t_out=16384, slabs=[(512, 1, 0, 16384)], c_out=128, act="none",
                   layout="rows_f32", c_valid=66))
    cs.append(Case("iter_fc1", "production", 256, n=1, v=1, t_out=4096, slabs=[(4352, 1, 0, 4096), (192, 1, 0, 4096)],
                   c_out=512, act="none"))
    cs.append(Case("iter_fc2", "production", 256, n=1, v=1, t_out=4096, slabs=[(512, 1, 0, 4096)], c_out=512, act="none"))
    cs.append(Case("iter_decpose", "production", 64, n=1, v=1, t_out=4096, slabs=[(512, 1, 0, 4096)], c_out=192,
                   act="none", layout="rows_f32", c_valid=132))
    for t in (64, 128):
        to = (t - 1) // 2 + 1
        cs.append(Case(f"b2_T{t}", "production", "ts", n=8, t_out=to, slabs=_taps(128, 2, t) + [(64, 2, 0, t)], c_out=128))
        cs.append(Case(f"b5_T{t}", "production", "ts", n=8, t_out=to, slabs=_taps(128, 2, t) + [(128, 2, 0, t)], c_out=128))
        cs.append(Case(f"b6_T{t}", "production", 256, n=8, t_out=to, slabs=_taps(256, 2, t) + [(128, 2, 0, t)], c_out=256))
    return cs


MATRIX = _case_matrix()
TS_CASES = [c for c in MATRIX if c.kern == "ts"]


@pytest.fixture
def clean_env(monkeypatch):
    """No tuning variable set: the prepared-launch cache is in use.  Tests set what they need on top."""
    for k in TUNING_VARS:
        monkeypatch.delenv(k, raising=False)
    return monkeypatch


def _rowgemm_kernels(fn):
    """Names of the rowgemm kernels `fn` launches (one torch.profiler pass with CUDA activities), spaces removed."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name.replace(" ", "") for e in prof.events() if "rowgemm" in e.name]


def _expected_kernel(case, kern):
    return f"rowgemm_ts_kernel<{ACT_CODE[case.act]}>" if kern == "ts" else f"rowgemm_umma_kernel<{kern},{ACT_CODE[case.act]}>"


def _device_inputs(case, seed):
    inp = case.inputs(seed)
    return {"slabs": [(a.cuda(), m, o) for a, m, o in inp["slabs"]], "w": inp["w"].cuda(), "bias": inp["bias"].cuda(),
            "res": None if inp["res"] is None else inp["res"].cuda()}


def _call(case, d, out):
    from temporal_inverse_kinematics_b200 import ops
    return ops.rowgemm(d["slabs"], d["w"], d["bias"], case.nv, case.v, case.t_out, act=case.act, slope=case.slope,
                       residual=d["res"], out_layout=case.layout, c_out_valid=case.c_valid, out=out)


def _guarded_out(case):
    """Output view with one guard slice either side, filled with a sentinel."""
    shape = case.out_shape()
    dt = torch.bfloat16 if case.bf16_out else torch.float32
    guard = torch.full((shape[0] + 2,) + shape[1:], 12345.0, dtype=dt, device="cuda")
    return guard, guard[1:-1]


def _bits(t):
    return t.view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32)


def _report(case, label, st):
    print(f"\n[bf16-rowgemm] family={case.family} case={case.name}{label} err/tol={st['ratio']:.4f} "
          f"need_c=2^-20*{st['need_c'] * 2 ** 20:.4f} mean_ulp={st['mean_ulp']:+.4f} toward_ulp={st['toward_ulp']:+.4f} "
          f"n_bias={st['n_bias']}")


def run_case(case, kern, label="", seed=0):
    """One call under the profiler, a second identical call, then: the kernel that ran, the guard slices, bitwise
    repeatability, and the comparator against fp64 (evaluated on the GPU)."""
    d = _device_inputs(case, seed)
    ref, scale = case.reference(d)
    guard, out = _guarded_out(case)
    ends = (guard[0].clone(), guard[-1].clone())
    names = _rowgemm_kernels(lambda: _call(case, d, out))
    want = _expected_kernel(case, kern)
    assert len(names) == 1 and want in names[0], (case.name, names, want)
    first = out.clone()
    _call(case, d, out)
    torch.cuda.synchronize()
    assert torch.equal(guard[0], ends[0]) and torch.equal(guard[-1], ends[1]), "write outside the output"
    assert torch.equal(_bits(out), _bits(first)), "two identical calls differ"
    st = compare(out, ref, scale, case.bf16_out)
    _report(case, label, st)
    assert verdict(st) == [], (case.name, label, st)
    return st


@pytest.mark.gpu
@pytest.mark.parametrize("case", MATRIX, ids=repr)
def test_bf16_rowgemm_matches_fp64(case, clean_env):
    run_case(case, case.kern)


@pytest.mark.gpu
@pytest.mark.parametrize("case", TS_CASES, ids=repr)
def test_bf16_rowgemm_without_ts_matches_fp64(case, clean_env):
    """Every weight-stationary case again on the SS kernel (TIK_NO_TS): both must agree with fp64."""
    clean_env.setenv("TIK_NO_TS", "1")
    run_case(case, case.c_out, label="[no_ts]")


OPT_SHAPES = {
    # one N tile (BN = 64), per-node bias keeps it off the TS kernel: every (option, group) pair fits
    "single_n_tile": Case("opt_single", "cost_model", 64, n=2, t_out=32, slabs=_taps(64, 1, 32) + [(64, 1, 0, 32)],
                          c_out=64, per_node=True),
    # five N tiles of 64: resident weights (options 0, 1) do not apply
    "multi_n_tile": Case("opt_multi", "cost_model", 64, n=2, t_out=32, slabs=_taps(64, 1, 32) + [(64, 1, 0, 32)],
                         c_out=320),
}
# (shape, option, group) with no plan: resident weights with several N tiles, and streamed weights with two staging
# tiles at four chunks per stage (two stages of 4 x 24 KB do not fit beside two 16 KB staging tiles)
OPT_REFUSED = {("multi_n_tile", o, g) for o in (0, 1) for g in (1, 2, 4)} | {(s, 2, 4) for s in OPT_SHAPES}


@pytest.mark.gpu
@pytest.mark.parametrize("shape", sorted(OPT_SHAPES))
@pytest.mark.parametrize("opt", [0, 1, 2, 3])
@pytest.mark.parametrize("group", [1, 2, 4])
def test_bf16_rowgemm_cost_model_options(shape, opt, group, clean_env):
    """TIK_UMMA_OPT forces (resident weights, staging tiles) = (1,2) (1,1) (0,2) (0,1); TIK_UMMA_GROUP the K chunks
    per ring stage.  A forced combination that does not fit is refused by name, before any launch."""
    case = OPT_SHAPES[shape]
    clean_env.setenv("TIK_UMMA_OPT", str(opt))
    clean_env.setenv("TIK_UMMA_GROUP", str(group))
    if (shape, opt, group) in OPT_REFUSED:
        d = _device_inputs(case, 0)
        with pytest.raises(RuntimeError, match="no shared-memory plan with TIK_UMMA_OPT"):
            _call(case, d, None)
        return
    run_case(case, case.kern, label=f"[opt{opt}_group{group}]")


@pytest.mark.gpu
@pytest.mark.parametrize("group", [1, 2, 4])
def test_bf16_rowgemm_ts_ring_groups(group, clean_env):
    """The TS kernel honours TIK_UMMA_GROUP and ignores TIK_UMMA_OPT."""
    clean_env.setenv("TIK_UMMA_OPT", "0")
    clean_env.setenv("TIK_UMMA_GROUP", str(group))
    case = next(c for c in MATRIX if c.name == "ktot512")
    run_case(case, "ts", label=f"[group{group}]")


# ------------------------------------------------------------------------------------------------ GPU: cache and capture
@pytest.mark.gpu
def test_prepared_launch_cache_eviction(clean_env):
    """34 distinct descriptors (the cache keeps 32), then the first again: evicted, prepared anew, still right."""
    cases = [Case(f"evict{i}", "cache", "ts" if i % 2 == 0 else 64, n=1, v=3, t_out=i + 1, slabs=_taps(64, 1, i + 1),
                  c_out=64, per_node=i % 2 == 1) for i in range(34)]
    kept = []
    for case in cases:
        d = _device_inputs(case, seed=len(kept))
        _, out = _guarded_out(case)
        _call(case, d, out)
        ref, scale = case.reference(d)
        assert verdict(compare(out, ref, scale, True)) == [], case.name
        kept.append((case, d, out, out.clone(), ref, scale))
    case, d, out, first, ref, scale = kept[0]
    out.fill_(7.0)
    _call(case, d, out)
    torch.cuda.synchronize()
    assert torch.equal(_bits(out), _bits(first))
    assert verdict(compare(out, ref, scale, True)) == []


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["residual_c128", "ktot512", "rows_f32_66_of_128"])
def test_cached_launch_follows_new_contents(name, clean_env):
    """Same addresses, new weight / bias / input / residual contents: the cached launch must read the new values."""
    case = next(c for c in MATRIX if c.name == name)
    d = _device_inputs(case, seed=0)
    _, out = _guarded_out(case)
    _call(case, d, out)
    new = case.inputs(seed=1)
    for (a, _, _), (b, _, _) in zip(d["slabs"], new["slabs"]):
        a.copy_(b)
    for k in ("w", "bias", "res"):
        if d[k] is not None:
            d[k].copy_(new[k])
    _call(case, d, out)
    torch.cuda.synchronize()
    ref, scale = case.reference(d)
    assert verdict(compare(out, ref, scale, case.bf16_out)) == []


@pytest.mark.gpu
def test_cuda_graph_capture_of_the_iterative_head(clean_env):
    """fc1 -> fc2 -> decpose into preallocated outputs, captured after an eager warm-up as the iterative head does:
    replay is bit-identical to eager and picks up new input contents."""
    from temporal_inverse_kinematics_b200 import ops
    m = 256
    g = torch.Generator().manual_seed(11)
    feat = torch.randn(1, m, 4352, generator=g).bfloat16().cuda()
    slab = torch.randn(1, m, 192, generator=g).bfloat16().cuda()
    w1 = (torch.randn(512, 4544, generator=g) / 4544 ** 0.5).bfloat16().cuda()
    w2 = (torch.randn(512, 512, generator=g) / 512 ** 0.5).bfloat16().cuda()
    w3 = (torch.randn(192, 512, generator=g) / 512 ** 0.5).bfloat16().cuda()
    b1, b2, b3 = (torch.randn(1, n, generator=g).cuda() for n in (512, 512, 192))
    h1 = torch.empty(1, m, 512, dtype=torch.bfloat16, device="cuda")
    h2 = torch.empty_like(h1)
    dd = torch.empty(m, 132, device="cuda")

    def body():
        ops.rowgemm([(feat, 1, 0), (slab, 1, 0)], w1, b1, 1, 1, m, out=h1)
        ops.rowgemm([(h1, 1, 0)], w2, b2, 1, 1, m, out=h2)
        ops.rowgemm([(h2, 1, 0)], w3, b3, 1, 1, m, out_layout="rows_f32", c_out_valid=132, out=dd)

    def check_against_fp64():
        r1, s1 = reference([(feat, 1, 0), (slab, 1, 0)], w1, b1, 1, 1, m, with_scale=True)
        assert verdict(compare(h1, r1, s1, True)) == []
        r2, s2 = reference([(h1, 1, 0)], w2, b2, 1, 1, m, with_scale=True)
        assert verdict(compare(h2, r2, s2, True)) == []
        r3, s3 = reference([(h2, 1, 0)], w3, b3, 1, 1, m, out_layout="rows_f32", c_out_valid=132, with_scale=True)
        assert verdict(compare(dd, r3, s3, False)) == []

    body()
    torch.cuda.synchronize()
    eager = dd.clone()
    check_against_fp64()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        body()
    dd.fill_(0.0)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(_bits(dd), _bits(eager))
    feat.copy_(torch.randn(1, m, 4352, generator=g).bfloat16())
    slab.copy_(torch.randn(1, m, 192, generator=g).bfloat16())
    graph.replay()
    torch.cuda.synchronize()
    replayed = (h1.clone(), dd.clone())
    assert not torch.equal(_bits(dd), _bits(eager))
    check_against_fp64()
    body()
    torch.cuda.synchronize()
    assert torch.equal(_bits(h1), _bits(replayed[0])) and torch.equal(_bits(dd), _bits(replayed[1]))


# ------------------------------------------------------------------------------------------------ GPU: refused calls
def _bad_calls():
    def base(nv=34, v=17, t=8, c=64, c_out=64, t_mul=1, bias_rows=1):
        g = torch.Generator().manual_seed(0)
        a = torch.randn(nv, t * t_mul, c, generator=g).bfloat16().cuda()
        w = torch.randn(c_out, c, generator=g).bfloat16().cuda()
        b = torch.randn(bias_rows, c_out, generator=g).cuda()
        return dict(slabs=[(a, t_mul, 0)], w=w, bias=b, nv=nv, v=v, t_out=t)

    def unaligned():
        k = base()
        a = k["slabs"][0][0]
        buf = torch.empty(a.numel() + 1, dtype=torch.bfloat16, device="cuda")
        view = buf[1:].view(a.shape)
        view.copy_(a)
        k["slabs"] = [(view, 1, 0)]
        return k

    def stem():
        k = base()
        x = torch.randn(2, 8, 17, 3, device="cuda")
        rw = torch.randn(17, 64, 3, device="cuda")
        k["stem_residual"] = (x, rw, 1)
        return k

    return {
        "c_out_not_multiple_of_64": (lambda: base(c_out=96), "c_out=96 must be a multiple of 64"),
        "slab_c_not_multiple_of_64": (lambda: base(c=96), "slab 0 malformed"),
        "t_mul_above_8": (lambda: base(t_mul=9), "slab 0 malformed"),
        "slab_base_not_16_byte_aligned": (unaligned, "16-byte aligned"),
        "stem_residual": (stem, "TIK_RES_STEM is only implemented by the fp32 kernel"),
        "bias_table_too_large": (lambda: base(nv=32, v=32, c_out=1024, bias_rows=32), "bias table too large"),
    }


BAD_CALLS = _bad_calls()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(BAD_CALLS))
def test_bf16_rowgemm_refuses_without_launching(name, clean_env):
    from temporal_inverse_kinematics_b200 import ops
    make, message = BAD_CALLS[name]
    k = make()
    c_out, nv, t_out = k["w"].shape[0], k["nv"], k["t_out"]
    out = torch.full((nv, t_out, c_out), 3.0, dtype=torch.bfloat16, device="cuda")
    errors = []

    def call():
        try:
            ops.rowgemm(out=out, **k)
        except RuntimeError as e:
            errors.append(str(e))

    assert _rowgemm_kernels(call) == []
    assert len(errors) == 1 and message in errors[0], errors
    assert bool((out == 3.0).all())
