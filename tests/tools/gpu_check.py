"""Step-by-step GPU diagnostics (run on the B200 box; each stage in its own process via tests/tools/gpu_check.sh).

    python tests/tools/gpu_check.py simt | umma | fused | net
"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import packed_emulator  # noqa: E402
from oracle import fk_port, geometry_port as gp, stgcn_port as sp, synth  # noqa: E402
from temporal_inverse_kinematics_b200 import _lib, engine, ops  # noqa: E402


def report(name, got, want, tol):
    got, want = got.float().cpu(), want.float().cpu()
    err = (got - want).abs()
    bad = err > tol
    status = "OK " if not bool(bad.any()) and bool(torch.isfinite(got).all()) else "FAIL"
    print(f"[{status}] {name}: max err {float(err.max()):.3e} (tol {tol:g}), ref absmax {float(want.abs().max()):.3e}, "
          f"bad {int(bad.sum())}/{bad.numel()}, nonfinite {int((~torch.isfinite(got)).sum())}", flush=True)
    if status == "FAIL" and got.dim() >= 2:
        e2 = err.reshape(-1, err.shape[-1])
        rows = (e2 > tol).any(1).nonzero().flatten()
        cols = (e2 > tol).any(0).nonzero().flatten()
        print(f"       bad rows {rows[:24].tolist()}{'...' if len(rows) > 24 else ''} ({len(rows)}/{e2.shape[0]}), "
              f"bad cols {cols[:24].tolist()}{'...' if len(cols) > 24 else ''} ({len(cols)}/{e2.shape[1]})")
        r = int(rows[0]) if len(rows) else 0
        print("       got ", got.reshape(-1, got.shape[-1])[r, :8].tolist())
        print("       want", want.reshape(-1, want.shape[-1])[r, :8].tolist())
    return status == "OK "


def stage_simt():
    from temporal_inverse_kinematics_b200 import geometry as G, kornia_geometry_conversion as KG, smpl_util as SU
    print("device", torch.cuda.get_device_name(0), "libtik", _lib.lib().tik_version())
    _lib.check(_lib.lib().tik_check_device())
    rs = np.random.RandomState(0)
    M = 1000
    x6 = rs.standard_normal((M, 6)).astype(np.float32)
    aa = rs.standard_normal((M, 3)).astype(np.float32)
    ok = report("rot6d", G.rot6d_to_rotmat(torch.from_numpy(x6).cuda()), torch.from_numpy(gp.rot6d_to_rotmat(x6)), 1e-5)
    ok &= report("aa->R kornia", KG.angle_axis_to_rotation_matrix(torch.from_numpy(aa).cuda()), torch.from_numpy(gp.angle_axis_to_rotation_matrix(aa)), 1e-5)
    R9 = gp.batch_rodrigues(aa)
    ok &= report("rodrigues", G.batch_rodrigues(torch.from_numpy(aa).cuda()), torch.from_numpy(R9), 1e-5)
    ok &= report("R->aa", G.rotation_matrix_to_angle_axis(torch.from_numpy(R9.reshape(-1, 3, 3)).cuda()), torch.from_numpy(gp.rotation_matrix_to_angle_axis(R9.reshape(-1, 3, 3))), 1e-4)
    F = 500
    pose = synth.make_axis_angles(F)
    rest = synth.make_rest_skeleton()
    j, lr, gr = SU.fk_body(torch.from_numpy(pose).cuda(), rest, synth.SMPLX_BODY_PARENTS, want_local=True, want_global=True)
    ej, eR, egR = fk_port.fk_from_axis_angle(pose.astype(np.float64), rest.astype(np.float64), synth.SMPLX_BODY_PARENTS)
    ok &= report("fk joints", j, torch.from_numpy(ej), 1e-4)
    ok &= report("fk local R", lr, torch.from_numpy(eR), 1e-4)
    ok &= report("fk global R", gr, torch.from_numpy(egR), 1e-4)
    # fp32 primitives
    N, V, T, Cc = 3, 17, 11, 64
    x = torch.randn(N, V, T, Cc, device="cuda")
    A = torch.rand(2, V, V, device="cuda") * (torch.rand(2, V, V, device="cuda") > 0.5)
    ok &= report("aggregate f32", ops.aggregate(x, A), torch.einsum("kvw,nvtc->knwtc", A, x), 1e-5)
    xb = x.bfloat16()
    ok &= report("aggregate bf16", ops.aggregate(xb, A), torch.einsum("kvw,nvtc->knwtc", A, xb.float()), 5e-2)
    w = torch.randn(128, 3 * Cc, device="cuda") * 0.1
    b = torch.randn(V, 128, device="cuda")
    h = x.view(N * V, T, Cc)
    y = ops.rowgemm([(h, 2, -1), (h, 2, 0), (h, 2, 1)], w, b, N * V, V, 6, act="relu")
    want = packed_emulator.rowgemm([(h.cpu(), 2, -1), (h.cpu(), 2, 0), (h.cpu(), 2, 1)], w.cpu(), b.cpu(), V, 6, "relu")
    ok &= report("rowgemm f32 3 taps stride 2", y, want, 1e-4)
    # fp32 network
    from temporal_inverse_kinematics_b200.pose_regressor import PoseRegressor, default_hparams
    m = PoseRegressor(default_hparams()).eval()
    sd = synth.make_regressor_state(sp.build_adjacency("coco", "uniform", 2, 1), seed=0)
    m.load_state_dict(sd)
    m = m.cuda()
    for (n, t) in [(3, 9), (2, 64)]:
        xx = synth.make_clips(n, t, seed=7)
        ok &= report(f"fp32 net n={n} t={t}", m(xx.cuda())["poses"], sp.regressor_forward(sd, xx)["poses"], 1e-4)
    return ok


def umma_case(name, nv, v, t_in, t_out, cs, c_out, t_mul, offs, act="relu", residual=False, layout="node", seed=0, tol=3e-2):
    g = torch.Generator().manual_seed(seed)
    slabs_cpu = [(torch.randn(nv, t_in, c, generator=g).bfloat16(), t_mul, o) for c, o in zip(cs, offs)]
    ktot = sum(cs)
    w = (torch.randn(c_out, ktot, generator=g) / np.sqrt(ktot)).bfloat16()
    b = torch.randn(v, c_out, generator=g)
    res = torch.randn(nv, t_out, c_out, generator=g).bfloat16() if residual else None
    want = packed_emulator.rowgemm(slabs_cpu, w, b, v, t_out, act, res)
    slabs = [(a.cuda(), m, o) for a, m, o in slabs_cpu]
    y = ops.rowgemm(slabs, w.cuda(), b.cuda(), nv, v, t_out, act=act, residual=None if res is None else res.cuda(), out_layout=layout)
    torch.cuda.synchronize()
    if layout == "time":
        want = want.view(nv // v, v, t_out, c_out).permute(0, 2, 1, 3)
    return report(name, y.reshape(want.shape), want, tol)


def stage_umma():
    ok = True
    # 1. plain GEMM, one K chunk, identity-like weights to expose layout errors
    nv, t = 1, 128
    a = torch.zeros(nv, t, 64)
    a[0, torch.arange(128), torch.arange(128) % 64] = 1.0
    a[0, :, 0] += torch.arange(128) / 128.0
    w = torch.zeros(64, 64)
    w[torch.arange(64), torch.arange(64)] = 1.0
    w[:, 1] += torch.arange(64) / 64.0
    b = torch.zeros(1, 64)
    want = packed_emulator.rowgemm([(a.bfloat16(), 1, 0)], w.bfloat16(), b, 1, t, "none")
    y = ops.rowgemm([(a.bfloat16().cuda(), 1, 0)], w.bfloat16().cuda(), b.cuda(), nv, 1, t, act="none")
    torch.cuda.synchronize()
    ok &= report("umma identity 128x64x64", y, want, 1e-2)
    ok &= umma_case("umma 1 tile K=64 N=64", 1, 1, 128, 128, [64], 64, 1, [0], act="none")
    ok &= umma_case("umma 1 tile K=128 N=128", 1, 1, 128, 128, [128], 128, 1, [0], act="none")
    ok &= umma_case("umma 3 tiles K=256 N=256", 1, 1, 300, 300, [256], 256, 1, [0], act="leaky")
    ok &= umma_case("umma K=4352 N=512 (head1)", 1, 1, 200, 200, [4352], 512, 1, [0], act="leaky")
    ok &= umma_case("umma node-major T=64 VV=2", 34, 17, 64, 64, [64], 64, 1, [0])
    ok &= umma_case("umma T=9 VV=14", 34, 17, 9, 9, [64], 128, 1, [0])
    ok &= umma_case("umma 3 taps stride 1", 34, 17, 64, 64, [64, 64, 64], 64, 1, [-1, 0, 1], residual=True)
    ok &= umma_case("umma 3 taps stride 2 + res slab", 34, 17, 64, 32, [128, 128, 128, 64], 128, 2, [-1, 0, 1, 0])
    ok &= umma_case("umma 3 taps stride 2 odd T=9->5", 51, 17, 9, 5, [128, 128, 128], 128, 2, [-1, 0, 1])
    ok &= umma_case("umma 5 taps T=11", 34, 17, 11, 11, [64] * 5, 64, 1, [-2, -1, 0, 1, 2])
    ok &= umma_case("umma time-major out", 34, 17, 8, 4, [256, 256, 256], 256, 2, [-1, 0, 1], layout="time")
    ok &= umma_case("umma T=200 > 128", 17, 17, 200, 200, [64, 64, 64], 64, 1, [-1, 0, 1])
    return ok


def stage_fused():
    """Fused graph conv (aggregation as a block-structured MMA with an MN-major B operand) vs a torch emulation."""
    ok = True
    V = 17
    for (n, t, cin, cout) in [(2, 7, 64, 64), (3, 64, 64, 64), (2, 9, 64, 128), (3, 32, 128, 128), (2, 16, 128, 256), (4, 5, 128, 128),
                              (2, 3, 64, 64), (150, 64, 64, 128)]:
        g = torch.Generator().manual_seed(n * 1000 + t)
        x = torch.randn(n, V, t, cin, generator=g).bfloat16()
        A = (torch.rand(1, V, V, generator=g) * (torch.rand(1, V, V, generator=g) > 0.6)).float()
        w = (torch.randn(cout, cin, generator=g) / np.sqrt(cin)).bfloat16()
        b = torch.randn(V, cout, generator=g)
        abd = ops.build_abd(A, t)
        y = ops.gcn_fused(x.cuda(), abd.cuda(), w.cuda(), b.cuda())
        torch.cuda.synchronize()
        Ab = A[0].bfloat16().float()                                      # the kernel sees bf16 adjacency entries
        xa = torch.einsum("vw,nvtc->nwtc", Ab, x.float()).bfloat16().float()
        want = torch.relu(torch.einsum("nwtc,oc->nwto", xa, w.float()) + b.view(1, V, 1, cout))
        ok &= report(f"fused gcn n={n} t={t} {cin}->{cout}", y, want, 6e-2)
    return ok


def stage_net():
    from temporal_inverse_kinematics_b200.pose_regressor import PoseRegressor, default_hparams
    ok = True
    sd = synth.make_regressor_state(sp.build_adjacency("coco", "uniform", 2, 1), seed=0)
    m = PoseRegressor(default_hparams()).eval()
    m.load_state_dict(sd)
    mc = PoseRegressor(default_hparams()).eval()
    mc.load_state_dict(sd)
    packed_cpu = engine.PackedNet(mc.backbone, mc._head(), "bf16")
    m = m.cuda().set_compute_dtype("bf16")
    for (n, t) in [(3, 9), (4, 64), (2, 13)]:
        xx = synth.make_clips(n, t, seed=7)
        y = m(xx.cuda())["poses"]
        torch.cuda.synchronize()
        ok &= report(f"bf16 net vs oracle n={n} t={t}", y, sp.regressor_forward(sd, xx)["poses"], 0.08)
        ok &= report(f"bf16 net vs bf16 emulation n={n} t={t}", y, packed_emulator.forward(packed_cpu, xx), 0.03)
    # quick timing, both dtypes
    for dt, n in [("fp32", 256), ("bf16", 256), ("bf16", 4096)]:
        m.set_compute_dtype(dt)
        x = synth.make_clips(n, 64, seed=3).cuda()
        for _ in range(2):
            m(x)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        reps = 5
        for _ in range(reps):
            m(x)
        torch.cuda.synchronize()
        dtm = (time.perf_counter() - t0) / reps
        print(f"[time] {dt} B={n} T=64: {dtm * 1e3:.2f} ms/batch = {n * 64 / dtm / 1e6:.2f} M frames/s", flush=True)
    return ok


if __name__ == "__main__":
    stage = sys.argv[1]
    ok = {"simt": stage_simt, "umma": stage_umma, "net": stage_net, "fused": stage_fused}[stage]()
    print(f"stage {stage}: {'PASS' if ok else 'FAIL'}")
    sys.exit(0 if ok else 1)
