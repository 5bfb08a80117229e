"""fp64 evaluation of the TikRowGemm definition (include/tik.h), shared by the fp32 and bf16 tik_rowgemm tests.

    out[row, :] = act( sum_slabs A_s[row_s, :] . W[:, koff_s:koff_s+c_s]^T + bias + residual )

A row is (row group nv = clip*V + node, frame t); slab s reads frame t*t_mul + t_off of its source, zero outside
[0, t_in).  Works on whatever device the inputs live on (CPU for small cases, the GPU's fp64 units for head-sized ones).

compare / verdict are the per-element comparator of a kernel result against this reference: |got - ref| <= R_BF16 |ref|
+ C_ACC S, plus a rounding-bias check (error model and measurement: tests/test_bf16_rowgemm.py).  The tik_rowgemm tests
and the per-block plan tests (tests/test_gpu_plan_blocks.py) share it.
"""
import torch

R_BF16 = 2.0 ** -8            # half a bf16 ulp, relative: the output rounding
C_ACC = 2.0 ** -20            # fp32 accumulation error relative to S
BIAS_MAX_ULP = 0.1
BIAS_MIN_ELEMS = 4096


def gather(a, t_out, t_mul, t_off):
    """a (NV, t_in, c) -> (NV, t_out, c) fp64: source frame t*t_mul + t_off, zero outside [0, t_in)."""
    nv, t_in, c = a.shape
    ts = torch.arange(t_out, device=a.device) * t_mul + t_off
    ok = (ts >= 0) & (ts < t_in)
    rows = torch.zeros(nv, t_out, c, dtype=torch.float64, device=a.device)
    rows[:, ok] = a.double()[:, ts[ok]]
    return rows


def to_layout(x, nv, v, t_out, out_layout="node", c_out_valid=None):
    """Node-major (NV, t_out, c_out) -> the shape tik_rowgemm writes for `out_layout`."""
    if out_layout == "node":
        return x
    if out_layout == "time":
        return x.view(nv // v, v, t_out, x.shape[-1]).permute(0, 2, 1, 3)
    if out_layout == "rows_f32":
        return x.reshape(nv * t_out, x.shape[-1])[:, : x.shape[-1] if c_out_valid is None else c_out_valid]
    raise ValueError(out_layout)


def reference(slabs, w, bias, nv, v, t_out, act="none", slope=0.01, residual=None, out_layout="node", c_out_valid=None,
              with_scale=False, gather_fn=gather):
    """slabs [(a (NV, t_in, c), t_mul, t_off)], w (c_out, sum c), bias (1 | v, c_out) (row nv uses bias[nv % v]),
    residual (NV, t_out, c_out) or None -> fp64 result in the output layout.

    with_scale=True also returns S = sum_k |a_k w_k| + |bias| + |residual| per output element, the magnitude an
    fp32 accumulation of the same terms has to be measured against."""
    c_out = w.shape[0]
    wd = w.double()
    acc = torch.zeros(nv, t_out, c_out, dtype=torch.float64, device=w.device)
    scale = torch.zeros_like(acc) if with_scale else None
    koff = 0
    for a, t_mul, t_off in slabs:
        c = a.shape[2]
        rows = gather_fn(a, t_out, t_mul, t_off)
        ws = wd[:, koff:koff + c]
        acc += rows @ ws.t()
        if with_scale:
            scale += rows.abs() @ ws.abs().t()
        koff += c
    b = bias.double().reshape(-1, c_out)
    b = b[torch.arange(nv, device=b.device) % v][:, None, :] if b.shape[0] > 1 else b[0]
    acc += b
    if with_scale:
        scale += b.abs()
    if residual is not None:
        acc += residual.double()
        if with_scale:
            scale += residual.double().abs()
    if act == "relu":
        acc = acc.clamp_min(0)
    elif act == "leaky":
        acc = torch.where(acc > 0, acc, acc * slope)
    elif act != "none":
        raise ValueError(act)
    out = to_layout(acc, nv, v, t_out, out_layout, c_out_valid)
    if not with_scale:
        return out
    return out, to_layout(scale, nv, v, t_out, out_layout, c_out_valid)


def ulp_bf16(x):
    """Spacing of bf16 numbers at |x| (x = m 2^e with 0.5 <= |m| < 1: eight significant bits -> 2^(e-8))."""
    _, e = torch.frexp(x)
    return torch.ldexp(torch.ones_like(x), e - 8)


def compare(got, ref, scale, bf16_out):
    """-> dict: ratio = max |got - ref| / tol, need_c = the smallest c that passes, and the rounding-bias means (in
    bf16 ulps) over the well-conditioned elements."""
    got, ref, scale = got.double(), ref.double(), scale.double()
    r = R_BF16 if bf16_out else 0.0
    err = (got - ref).abs()
    tol = r * ref.abs() + C_ACC * scale
    ratio = torch.where(tol > 0, err / tol.clamp_min(1e-300), torch.where(err > 0, torch.inf, 0.0))
    excess = (err - r * ref.abs()).clamp_min(0)
    need_c = torch.where(scale > 0, excess / scale.clamp_min(1e-300), torch.where(excess > 0, torch.inf, 0.0))
    st = {"ratio": float(ratio.max()) if ratio.numel() else 0.0, "need_c": float(need_c.max()) if need_c.numel() else 0.0,
          "finite": bool(torch.isfinite(got).all()), "n_bias": 0, "mean_ulp": 0.0, "toward_ulp": 0.0}
    if bf16_out:
        u = ulp_bf16(ref)
        well = (ref != 0) & (C_ACC * scale <= u / 16)
        st["n_bias"] = int(well.sum())
        if st["n_bias"]:
            d = ((got - ref) / u)[well]
            st["mean_ulp"] = float(d.mean())
            st["toward_ulp"] = float((d * ref.sign()[well]).mean())
    return st


def verdict(st):
    """Reasons the comparator rejects a result (empty: accepted)."""
    bad = []
    if not st["finite"]:
        bad.append("non-finite output")
    if not st["ratio"] <= 1.0:
        bad.append(f"max err/tol {st['ratio']:.3g}")
    if st["n_bias"] >= BIAS_MIN_ELEMS and (abs(st["mean_ulp"]) >= BIAS_MAX_ULP or abs(st["toward_ulp"]) >= BIAS_MAX_ULP):
        bad.append(f"rounding bias {st['mean_ulp']:+.3f} / {st['toward_ulp']:+.3f} ulp")
    return bad
