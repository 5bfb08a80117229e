"""Test-only torch (CPU) emulation of the kernel sequence of csrc/plan.cu over a PackedNet.

Mirrors what the CUDA kernels compute from the *packed* tensors (node-major layout, aggregate-first graph
convolution, slab-wise implicit GEMM with zero padding), so that the eval-mode folding in
temporal_inverse_kinematics_b200/engine.py can be checked against the oracle without a GPU.
Never used by the product path.
"""
import torch


def _slab(a, t_out, t_mul, t_off):
    """a (NV, t_in, c) -> (NV, t_out, c): frame t_out*t_mul + t_off, zeros outside [0, t_in)."""
    nv, t_in, c = a.shape
    idx = torch.arange(t_out) * t_mul + t_off
    ok = (idx >= 0) & (idx < t_in)
    out = a.new_zeros((nv, t_out, c))
    out[:, ok] = a[:, idx[ok]]
    return out


def rowgemm(slabs, w, bias, v, t_out, act, residual=None, quant=None):
    a = torch.cat([_slab(s, t_out, m, o) for s, m, o in slabs], dim=-1).float()
    y = a @ w.float().t()
    nv = a.shape[0]
    if bias.dim() == 2 and bias.shape[0] > 1:
        y = y + bias[torch.arange(nv) % v][:, None, :]
    else:
        y = y + bias.reshape(1, 1, -1)
    if residual is not None:
        y = y + residual.float()
    if act == "relu":
        y = torch.relu(y)
    elif act == "leaky":
        y = torch.nn.functional.leaky_relu(y, 0.01)
    return y if quant is None else y.to(quant)


def _hilo(a, q):
    """fp32 -> bf16 hi + bf16 lo (what the stem-block kernel feeds the tensor core), back in fp32."""
    hi = a.to(q).float()
    return hi + (a - hi).to(q).float()


def stem_block_applies(packed):
    """Mirror of stem_block_supported (csrc/stem_block.cu): the first block runs as one tensor-core kernel."""
    net = packed.net
    b = net.blocks[0]
    return (packed.tdtype == torch.bfloat16 and net.n_blocks > 1 and net.K == 1 and net.c_in == 3 and b.c_out == 64
            and b.kt == 3 and b.stride == 1 and net.V <= 17 and b.res_kind in (0, 2))   # V * 15 tile rows <= 256


def forward(packed, x):
    """x (N,T,V,C) fp32 CPU -> poses (N,T',head_out).  Activations are rounded to packed.tdtype between kernels."""
    t = packed.named
    q = packed.tdtype
    net = packed.net
    N, T, V, Cin = x.shape
    K = net.K
    x0 = x * t["in_scale"].view(1, 1, V, Cin) + t["in_shift"].view(1, 1, V, Cin)
    cur = None
    for i in range(net.n_blocks):
        b = net.blocks[i]
        A = t[f"b{i}.agg"]
        fused0 = i == 0 and stem_block_applies(packed)
        if i == 0:
            xa = torch.einsum("kvw,ntvc->ntwkc", A, x0).reshape(N, T, V, K * Cin)          # (n,t,w,k*Cin+ci)
            wg = t["b0.w_gcn"]
            if fused0:                                                                       # bf16 weights, hi/lo inputs
                xa, wg = _hilo(xa, q), wg.to(q).float()
            h = torch.relu(torch.einsum("ntwj,cj->ntwc", xa, wg) + t["b0.b_gcn"].view(1, 1, V, -1))
            h = h.permute(0, 2, 1, 3).reshape(N * V, T, b.c_out).to(q)
        else:
            xn = cur.view(N, V, T, b.c_in).float()
            xa = torch.einsum("kvw,nvtc->knwtc", A, xn).to(q).reshape(K, N * V, T, b.c_in)
            h = rowgemm([(xa[k], 1, 0) for k in range(K)], t[f"b{i}.w_gcn"], t[f"b{i}.b_gcn"], V, T, "relu", quant=q)
        pad = (b.kt - 1) // 2
        t_out = (T - 1) // b.stride + 1
        slabs = [(h, b.stride, dt - pad) for dt in range(b.kt)]
        residual = None
        if b.res_kind == 3:
            slabs.append((cur, b.stride, 0))
        elif b.res_kind == 1:
            residual = cur
        elif b.res_kind == 2:
            xs = x[:, torch.arange(t_out) * b.stride]                                        # raw input frames
            if fused0:
                # the kernel multiplies (s0 * x) hi/lo by the unscaled bf16 residual weights and keeps R0 in fp32 (TMEM)
                s0 = t["in_scale"].view(V, Cin)
                vb = s0.abs().argmax(dim=0)                                                  # per channel: node with the largest scale
                sc = s0[vb, torch.arange(Cin)]
                wr = t["b0.w_res_stem"][vb, :, torch.arange(Cin)].t().double() / sc.double()  # (Cout, Cin)
                wr = torch.where(sc[None, :] != 0, wr, torch.zeros_like(wr)).float().to(q).float()
                residual = torch.einsum("ci,ntvi->nvtc", wr, _hilo(xs * s0.view(1, 1, V, Cin), q)).reshape(N * V, t_out, b.c_out)
            else:
                residual = torch.einsum("vci,ntvi->nvtc", t["b0.w_res_stem"], xs).reshape(N * V, t_out, b.c_out).to(q)
        if fused0:                                                                           # taps only; R0 added in fp32
            w_taps = t["b0.w_tcn"][:, : b.kt * b.c_out]
            cur = rowgemm(slabs, w_taps, t["b0.b_tcn"], V, t_out, "relu", residual, quant=q)
            T = t_out
            continue
        if b.res_as_slab:                                                                    # identity block in w_tcn
            slabs.append((residual, 1, 0))
            residual = None
        cur = rowgemm(slabs, t[f"b{i}.w_tcn"], t[f"b{i}.b_tcn"], V, t_out, "relu", residual, quant=q)
        T = t_out
    feat = cur.view(N, V, T, -1).permute(0, 2, 1, 3).reshape(N * T, -1)
    if net.head_hidden == 0:
        return feat.view(N, T, -1).float()
    z = rowgemm([(feat[None], 1, 0)], t["w1"], t["b1"], 1, N * T, "leaky", quant=q)
    y = rowgemm([(z, 1, 0)], t["w2"], t["b2"], 1, N * T, "none")
    return y[0, :, :net.head_out].reshape(N, T, net.head_out)
