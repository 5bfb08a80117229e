"""Whole-batch timings of the bf16 implicit GEMM (ops.rowgemm) at layer shapes of the network.

    python tools/umma_probe.py grp [shape]   ring-stage grouping (TIK_UMMA_GROUP) x shared-memory option (TIK_UMMA_OPT)
    python tools/umma_probe.py fill          DRAM or the L2 -> shared-memory fill: which binds the temporal conv?
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from temporal_inverse_kinematics_b200 import ops  # noqa: E402


def bench(fn, reps=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


def grp():
    """Sweep the ring-stage grouping (TIK_UMMA_GROUP) and shared-memory option (TIK_UMMA_OPT) on whole-batch layer shapes."""
    V, n = 17, 4096
    g = torch.Generator(device="cuda").manual_seed(0)
    shapes = [("b1 tcn 64->64 T64 K=256", 64, 64, 64, 64, 1, 64),
              ("b2 tcn 128->128 s2 K=448", 64, 32, 128, 64, 2, 128),
              ("b3 tcn 128->128 T32 K=512", 32, 32, 128, 128, 1, 128),
              ("b6 tcn 256->256 s2 K=896", 16, 8, 256, 128, 2, 256)]
    only = sys.argv[2:] and int(sys.argv[2])
    for si, (name, t_in, t_out, ch, cres, stride, c_out) in enumerate(shapes):
        if sys.argv[2:] and si != only:
            continue
        nv = n * V
        h = torch.randn(nv, t_in, ch, device="cuda", generator=g).bfloat16()
        r = torch.randn(nv, t_in, cres, device="cuda", generator=g).bfloat16()
        slabs = [(h, stride, -1), (h, stride, 0), (h, stride, 1), (r, stride, 0)]
        w = (torch.randn(c_out, 3 * ch + cres, device="cuda", generator=g) * 0.05).bfloat16()
        b = torch.zeros(1, c_out, device="cuda")
        gb = (h.numel() * 2 + r.numel() * 2 + nv * t_out * c_out * 2) / 1e9
        ref = None
        for opt in ("", "0", "1", "2", "3"):
            for grp_ in ("1", "2", "4"):
                os.environ["TIK_UMMA_GROUP"] = grp_
                if opt:
                    os.environ["TIK_UMMA_OPT"] = opt
                else:
                    os.environ.pop("TIK_UMMA_OPT", None)
                try:
                    out = ops.rowgemm(slabs, w, b, nv, V, t_out, act="relu")
                    us = bench(lambda: ops.rowgemm(slabs, w, b, nv, V, t_out, act="relu"), reps=5)
                except RuntimeError as e:
                    print(f"{name} opt={opt or 'auto'} G={grp_}: {str(e)[:80]}", flush=True)
                    continue
                if ref is None:
                    ref = out
                same = bool((out == ref).all())
                print(f"{name} opt={opt or 'auto'} G={grp_}: {us:7.1f} us  {gb / us * 1e3:5.2f} TB/s  same={same}", flush=True)
        del h, r, w
    os.environ.pop("TIK_UMMA_GROUP", None)
    os.environ.pop("TIK_UMMA_OPT", None)


def fill():
    """Is the temporal conv bound by DRAM or by the L2 -> shared-memory fill?  Same K and fill bytes, different
    numbers of distinct tensors behind the four K slabs."""
    V, n = 17, 4096
    g = torch.Generator(device="cuda").manual_seed(0)
    nv = n * V
    for (T, C) in ((32, 128), (64, 64)):
        ts_ = [torch.randn(nv, T, C, device="cuda", generator=g).bfloat16() for _ in range(4)]
        w = (torch.randn(C, 4 * C, device="cuda", generator=g) * 0.05).bfloat16()
        b = torch.zeros(1, C, device="cuda")
        cases = {"3 taps + residual (2 tensors)": [(ts_[0], 1, -1), (ts_[0], 1, 0), (ts_[0], 1, 1), (ts_[1], 1, 0)],
                 "1 tensor x4 (same tap)": [(ts_[0], 1, 0)] * 4,
                 "4 distinct tensors": [(ts_[i], 1, 0) for i in range(4)]}
        for name, slabs in cases.items():
            us = bench(lambda: ops.rowgemm(slabs, w, b, nv, V, T, act="relu"), reps=8)
            distinct = len({id(s[0]) for s in slabs})
            gb = (distinct * nv * T * C * 2 + nv * T * C * 2) / 1e9
            print(f"T={T} C={C} {name}: {us:6.1f} us  DRAM {gb:.2f} GB -> {gb / us * 1e3:.2f} TB/s; fill {4 * nv * T * C * 2 / 1e9 / us * 1e3:.2f} TB/s", flush=True)


if __name__ == "__main__":
    modes = {"grp": grp, "fill": fill}
    if len(sys.argv) < 2 or sys.argv[1] not in modes:
        sys.exit(__doc__)
    modes[sys.argv[1]]()
