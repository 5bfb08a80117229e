"""tik_rowgemm in fp32 on the tensor pipe (csrc/rowgemm_tf32.cu: 3xTF32, per-chunk accumulation) against an fp64
evaluation of the TikRowGemm definition (include/tik.h): tap shifts, strides, zero padding, ragged row counts, per-node
bias, identity residual, every output layout, a guard region around the output -- and against the SIMT fp32 kernel."""
import os

import pytest
import torch

from rowgemm_reference import reference

pytestmark = pytest.mark.gpu
V = 17


CASES = [
    # n clips, t_in, t_out, [(c, t_mul, t_off)], c_out, act, per-node bias, residual, layout
    (2, 9, 9, [(64, 1, -1), (64, 1, 0), (64, 1, 1)], 64, "relu", False, True, "node"),        # 3 taps + identity residual, 306 rows
    (3, 32, 16, [(128, 2, -1), (128, 2, 0), (128, 2, 1), (64, 2, 0)], 128, "relu", False, False, "node"),   # stride 2 + residual conv slab
    (1, 13, 13, [(64, 1, 0)], 128, "relu", True, False, "node"),                              # graph-conv GEMM: per-node bias, 2 chunks
    (5, 4, 2, [(256, 2, -1), (256, 2, 0), (256, 2, 1), (256, 2, 0)], 256, "relu", False, False, "time"),   # last block: feature order
    (40, 16, 8, [(96, 2, 0)], 64, "none", False, False, "node"),                              # 3 chunks, 5440 rows: several tiles per SM slot
]


@pytest.mark.parametrize("case", CASES)
def test_tf32_rowgemm_matches_fp64(case):
    from temporal_inverse_kinematics_b200 import ops
    n, t_in, t_out, slab_cfg, c_out, act, per_node, with_res, layout = case
    nv = n * V
    g = torch.Generator().manual_seed(nv + t_in + c_out)
    slabs = [(torch.randn(nv, t_in, c, generator=g), m, o) for c, m, o in slab_cfg]
    ktot = sum(c for c, _, _ in slab_cfg)
    w = torch.randn(c_out, ktot, generator=g) / ktot ** 0.5
    bias = torch.randn(V if per_node else 1, c_out, generator=g)
    res = torch.randn(nv, t_out, c_out, generator=g) if with_res else None
    want = reference(slabs, w, bias, nv, V, t_out, act, 0.01, res, out_layout=layout)
    shape = (nv, t_out, c_out) if layout == "node" else (n, t_out, V, c_out)
    outs = {}
    for mode in ("tf32", "simt"):
        os.environ.pop("TIK_NO_TF32", None)
        if mode == "simt":
            os.environ["TIK_NO_TF32"] = "1"
        try:
            guard = torch.full((shape[0] + 2,) + shape[1:], 12345.0, device="cuda")   # one extra slice either side of the output
            out = guard[1:-1]
            ops.rowgemm([(a.cuda(), m, o) for a, m, o in slabs], w.cuda(), bias.cuda(), nv, V, t_out, act=act,
                        residual=None if res is None else res.cuda(), out_layout=layout, out=out)
            torch.cuda.synchronize()
        finally:
            os.environ.pop("TIK_NO_TF32", None)
        assert bool((guard[0] == 12345.0).all()) and bool((guard[-1] == 12345.0).all()), mode
        outs[mode] = out.cpu().double()
        err = float((outs[mode] - want).abs().max() / want.abs().max())
        assert err < 2e-6, (mode, err)
    assert float((outs["tf32"] - outs["simt"]).abs().max()) < 2e-5


def test_tf32_head_output_rows_f32():
    """Head Linear(512, 66): c_out = 66 (not a multiple of 4), 'rows_f32' layout with 66 valid columns, LeakyReLU off."""
    from temporal_inverse_kinematics_b200 import ops
    rows = 300
    g = torch.Generator().manual_seed(5)
    a = torch.randn(1, rows, 512, generator=g)
    w = torch.randn(66, 512, generator=g) / 512 ** 0.5
    b = torch.randn(1, 66, generator=g)
    guard = torch.full((rows + 2, 66), 777.0, device="cuda")
    out = guard[1:-1]
    ops.rowgemm([(a.cuda(), 1, 0)], w.cuda(), b.cuda(), 1, 1, rows, out_layout="rows_f32", c_out_valid=66, out=out)
    torch.cuda.synchronize()
    want = reference([(a, 1, 0)], w, b, 1, 1, rows, out_layout="rows_f32", c_out_valid=66)
    assert bool((guard[0] == 777.0).all()) and bool((guard[-1] == 777.0).all())
    assert float((out.cpu().double() - want).abs().max() / want.abs().max()) < 2e-6


def test_tf32_long_k_accumulation_does_not_drift():
    """The tensor core's fp32 accumulator truncates: with one accumulator for all of K the error grows linearly with K
    (3e-5 at K = 4352).  Per-chunk accumulation keeps the head GEMM at the 1e-6 level."""
    from temporal_inverse_kinematics_b200 import ops
    rows, k, n = 2048, 4352, 512
    g = torch.Generator(device="cuda").manual_seed(1)
    a = torch.randn(1, rows, k, device="cuda", generator=g).abs()          # same-sign products: the worst case for truncation
    w = torch.randn(n, k, device="cuda", generator=g).abs() / k
    b = torch.zeros(1, n, device="cuda")
    out = ops.rowgemm([(a, 1, 0)], w, b, 1, 1, rows)
    want = reference([(a, 1, 0)], w, b, 1, 1, rows)[0]
    assert float(((out[0].double() - want).abs() / want.abs()).max()) < 2e-6


def test_tf32_rowgemm_random_shapes():
    """Seeded sweep over ragged shapes: row counts that are not multiples of 128, output widths that are not multiples of
    64 / 4, one to four slabs with strides 1..3 and tap offsets, K from 32 to 544 -- each against fp64 with a guard region."""
    import random
    from temporal_inverse_kinematics_b200 import ops
    rnd = random.Random(1234)
    for case in range(24):
        n = rnd.choice([1, 2, 3, 9])
        v = rnd.choice([1, 5, 17])
        nv = n * v
        t_out = rnd.choice([1, 3, 8, 31, 64])
        t_mul = rnd.choice([1, 1, 2, 3])
        n_slabs = rnd.choice([1, 1, 2, 3, 4])
        c_out = rnd.choice([4, 40, 64, 72, 100, 128, 132, 256, 260])
        slabs = []
        g = torch.Generator().manual_seed(case)
        for _ in range(n_slabs):
            c = 32 * rnd.choice([1, 1, 2, 3, 4, 5])
            t_in = t_out * t_mul + rnd.choice([0, 1, 2])
            slabs.append((torch.randn(nv, t_in, c, generator=g), t_mul, rnd.choice([-2, -1, 0, 0, 1, 2])))
        ktot = sum(a.shape[2] for a, _, _ in slabs)
        w = torch.randn(c_out, ktot, generator=g) / ktot ** 0.5
        per_node = rnd.random() < 0.5
        bias = torch.randn(v if per_node else 1, c_out, generator=g)
        res = torch.randn(nv, t_out, c_out, generator=g) if rnd.random() < 0.5 else None
        act = rnd.choice(["none", "relu", "leaky"])
        acc = reference(slabs, w, bias, nv, v, t_out, act, 0.01, res)
        guard = torch.full((nv + 2, t_out, c_out), 4242.0, device="cuda")
        out = guard[1:-1]
        ops.rowgemm([(a.cuda(), m, o) for a, m, o in slabs], w.cuda(), bias.cuda(), nv, v, t_out, act=act, slope=0.01,
                    residual=None if res is None else res.cuda(), out=out)
        torch.cuda.synchronize()
        assert bool((guard[0] == 4242.0).all()) and bool((guard[-1] == 4242.0).all()), case
        err = float((out.cpu().double() - acc).abs().max() / acc.abs().max())
        assert err < 3e-6, (case, err, nv, t_out, c_out, ktot)
