"""Keypoint fitting throughput: smpl_util.fit_keypoints (one tik_fit_keypoints launch, COCO-17, translation fitted) at
F = 1,048,576 frames for n_iter in {1, 10, 30}, on a V = 10,475 synthetic SmplxBodyModel (pose-blended landmarks) and on
the synthetic full skeleton.  Targets are keypoints of random poses plus 1 cm of noise; the start is those poses plus
0.1 rad of noise.  CUDA events per call after warm-up; the inputs (~0.5 GB) do not fit in L2.

    python tools/bench_fit.py --out DIR [--frames F] [--steps N] [--warmup W]

FMAs per frame-iteration are counted from the shapes for an iteration whose step is accepted (the normal equations
are formed again only then): H as the kernel forms it (4 x 4 tiles of the lower triangle over 3n rows), g, the
Cholesky (P^3/6) and its two substitutions (P^2), one keypoint forward (Rodrigues, FK, pose blend, skinning) and the
Jacobian (ancestor blocks, landmark blocks with their pose-blend term).  The FP32-FMA bound is 148 SMs x 128 lanes x the
max SM clock.  Writes DIR/bench_fit.json (DIR is created; nothing is written elsewhere)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import smplx_synth  # noqa: E402
from temporal_inverse_kinematics_b200 import smpl_util as SU  # noqa: E402

PARENTS = SU.SMPLX_FULL_PARENTS[:55]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        name, power, clock = torch.cuda.get_device_name(0), "unknown", "unknown"
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def fmas_per_iteration(sel, L, skin_nnz, pose_blend, P=69):
    """FMAs of one accepted iteration of one frame, from the shapes."""
    n = len(sel)
    nt = (P + 3) // 4
    depth = [0] * 55
    for j, p in enumerate(PARENTS):
        depth[j] = 0 if p < 0 else depth[p] + 1
    H = 3 * n * nt * (nt + 1) // 2 * 16
    g = 3 * n * P
    chol = P ** 3 // 6 + P * P
    fwd = 22 * 30 + 55 * 36 + (3 * L * 21 * 9 if pose_blend else 0) + 3 * L * skin_nnz * 4 + 3 * n
    anc = sum(min(depth[q], 22) for q in sel if q < 55)                         # proper ancestors among joints 0..21
    jac = 22 * 36 + anc * 18 + (n - sum(q < 55 for q in sel)) * 22 * (skin_nnz * 13 + 9 + (108 + 27 if pose_blend else 0))
    return {"H": H, "g": g, "cholesky_and_substitutions": chol, "forward": fwd, "jacobian": jac,
            "total": H + g + chol + fwd + jac}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for bench_fit.json")
    ap.add_argument("--frames", type=int, default=1 << 20)
    ap.add_argument("--iters", default="1,10,30")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fit needs a GPU")
    info = gpu_info()
    try:
        clock_ghz = float(info["max_sm_clock"].split()[0]) / 1000.0
    except (ValueError, IndexError):
        clock_ghz = 1.965
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    fma_peak = sms * 128 * clock_ghz * 1e9
    mesh = SU.SmplxBodyModel(smplx_synth.make_smplx_arrays(10475, seed=0), skeleton="full")
    synth = SU.SyntheticBodyModel(skeleton="full")
    coco = SU.keypoint_indices("coco")
    F = args.frames
    gen = torch.Generator(device="cuda").manual_seed(F)
    theta = torch.randn(F, 22, 3, device="cuda", generator=gen) * 0.3
    tau = torch.randn(F, 3, device="cuda", generator=gen)
    init = theta + torch.randn(F, 22, 3, device="cuda", generator=gen) * 0.1
    betas = np.linspace(-1, 1, 10)
    results = []
    for name, model in (("mesh", mesh), ("synthetic", synth)):
        pack = model.keypoint_pack(torch.device("cuda"))
        nnz = int((pack.skin_w != 0).sum(1).max())
        y = SU.keypoints(theta, model, betas, tau) + torch.randn(F, 17, 3, device="cuda", generator=gen) * 0.01
        fmas = fmas_per_iteration(coco, pack.n_landmarks, nnz, pack.lm_posedirs is not None)
        for n_iter in [int(s) for s in args.iters.split(",")]:
            def run():
                return SU.fit_keypoints(y, model, init, betas, tau, "coco", None, 1e-3, n_iter)
            for _ in range(args.warmup):
                out = run()
            torch.cuda.synchronize()
            times = []
            for _ in range(args.steps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                out = run()
                e1.record()
                torch.cuda.synchronize()
                times.append(e0.elapsed_time(e1) * 1e-3)
            t = float(np.median(times))
            ratio = (out["cost"] / out["cost_init"]).float()
            bound = F * n_iter * fmas["total"] / fma_peak
            r = {"model": name, "frames": F, "n_iter": n_iter, "median_s": t, "min_s": min(times), "max_s": max(times),
                 "frames_per_s": F / t, "frame_iterations_per_s": F * n_iter / t, "fma_per_frame_iteration": fmas,
                 "share_of_fma_peak": bound / t, "median_cost_ratio": float(ratio.median())}
            results.append(r)
            print(f"{name:>9} n_iter={n_iter:3d}: {t * 1e3:9.2f} ms  {F / t / 1e6:7.3f} M frames/s  "
                  f"{r['share_of_fma_peak'] * 100:5.1f} % of the FP32-FMA bound  median cost ratio {r['median_cost_ratio']:.2e}",
                  flush=True)
        del y
    doc = {"tool": "tools/bench_fit.py", **info, "sms": sms, "fma_peak_per_s": fma_peak, "fma_counts_are_estimates": True,
           "steps": args.steps, "warmup": args.warmup, "select": "coco", "fit_transl": True, "prior_weight": 1e-3,
           "results": results}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_fit.json"), "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps({k: doc[k] for k in ("gpu", "power_limit", "max_sm_clock")}))


if __name__ == "__main__":
    main()
