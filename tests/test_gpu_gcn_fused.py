"""tik_gcn_fused (aggregation + channel GEMM + bias + ReLU in one tensor-core kernel) against a torch emulation that
rounds where the kernel rounds (bf16 adjacency, bf16 aggregate, fp32 accumulate), for every (Cin, Cout) variant --
including the transposed 256 -> 256 kernel (weights in tensor memory, output channels split over two CTAs)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n,t,cin,cout", [
    (2, 7, 64, 64), (3, 64, 64, 64), (2, 9, 64, 128), (3, 32, 128, 128), (2, 16, 128, 256), (4, 5, 128, 128),
    (150, 64, 64, 128),
    (3, 8, 256, 256),        # one wave, 4-frame tiles (the last block at T = 64)
    (1, 1, 256, 256),        # a single frame
    (2, 13, 256, 256),       # 5 + 5 + shifted 5 frames: overlapping last tile
    (3, 32, 256, 256),       # 5-frame tiles: 85 rows, N = 96 (the widest accumulator)
    (5, 16, 256, 256),       # the last block at T = 128
    (310, 8, 256, 256),      # 620 tiles x 2 halves over 148 CTAs: every ring / accumulator parity, ragged tail
])
def test_gcn_fused_matches_emulation(n, t, cin, cout):
    from temporal_inverse_kinematics_b200 import ops
    V = 17
    g = torch.Generator().manual_seed(n * 1000 + t + cin)
    x = torch.randn(n, V, t, cin, generator=g).bfloat16()
    A = (torch.rand(1, V, V, generator=g) * (torch.rand(1, V, V, generator=g) > 0.6)).float()
    w = (torch.randn(cout, cin, generator=g) / np.sqrt(cin)).bfloat16()
    b = torch.randn(V, cout, generator=g)
    y = ops.gcn_fused(x.cuda(), ops.build_abd(A, t, cin).cuda(), w.cuda(), b.cuda())
    torch.cuda.synchronize()
    Ab = A[0].bfloat16().float()
    if cin == 256:           # channel GEMM first, its result rounded to bf16, then the aggregation
        z = torch.einsum("nvtc,oc->nvto", x.float(), w.float()).bfloat16().float()
        want = torch.relu(torch.einsum("vw,nvto->nwto", Ab, z) + b.view(1, V, 1, cout))
    else:                    # aggregate rounded to bf16, then the channel GEMM
        xa = torch.einsum("vw,nvtc->nwtc", Ab, x.float()).bfloat16().float()
        want = torch.relu(torch.einsum("nwtc,oc->nwto", xa, w.float()) + b.view(1, V, 1, cout))
    err = (y.float().cpu() - want).abs()
    assert float(err.max()) < 6e-2 and float(err.pow(2).mean().sqrt()) < 6e-3, (float(err.max()), float(err.pow(2).mean().sqrt()))

