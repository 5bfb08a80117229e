"""fp64 evaluation of the TikRowGemm definition (include/tik.h), shared by the fp32 and bf16 tik_rowgemm tests.

    out[row, :] = act( sum_slabs A_s[row_s, :] . W[:, koff_s:koff_s+c_s]^T + bias + residual )

A row is (row group nv = clip*V + node, frame t); slab s reads frame t*t_mul + t_off of its source, zero outside
[0, t_in).  Works on whatever device the inputs live on (CPU for small cases, the GPU's fp64 units for head-sized ones).
"""
import torch


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
