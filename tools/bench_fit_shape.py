"""Shape fitting throughput: smpl_util.fit_keypoints_shape against smpl_util.fit_keypoints on the same data, alternating
in one process, at F = 1,048,576 frames (COCO-17, translation fitted) for n_iter in {1, 10, 30}, on a V = 10,475
synthetic SmplxBodyModel (pose-blended landmarks) and on the synthetic full skeleton, with the frames grouped as 1,024
sequences of 1,024 frames and as sequences of log-uniform lengths in [60, 3000].  Targets are keypoints of random poses
and a random shape per sequence plus 1 cm of noise; the start is those poses plus 0.1 rad of noise and the mean shape.
A 256 MB buffer is overwritten before every timed call, so no call starts from inputs left in L2.  CUDA events per call.

    python tools/bench_fit_shape.py --out DIR [--frames F] [--iters 1,10,30] [--steps N] [--warmup W]

Writes DIR/bench_fit_shape.json (DIR is created; nothing is written elsewhere)."""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_fit import gpu_info  # noqa: E402
from oracle import smplx_synth  # noqa: E402
from temporal_inverse_kinematics_b200 import _lib as L  # noqa: E402
from temporal_inverse_kinematics_b200 import smpl_util as SU  # noqa: E402

LAUNCHES_PER_ITERATION = 4          # frame, sequence, candidate and accept kernels
LAUNCHES_FIXED = 4                  # sequence init, start forward, initial cost, output


def layouts(F, seed):
    rs = np.random.RandomState(seed)
    out = {"1024x1024": [1024] * (F // 1024)}
    lens, left = [], F
    while left > 0:
        n = min(left, int(np.exp(rs.uniform(np.log(60), np.log(3000)))))
        lens.append(n)
        left -= n
    out["loguniform_60_3000"] = lens
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for bench_fit_shape.json")
    ap.add_argument("--frames", type=int, default=1 << 20)
    ap.add_argument("--iters", default="1,10,30")
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fit_shape needs a GPU")
    info = gpu_info()
    F = args.frames
    mesh = SU.SmplxBodyModel(smplx_synth.make_smplx_arrays(10475, seed=0), skeleton="full")
    synth = SU.SyntheticBodyModel(skeleton="full")
    gen = torch.Generator(device="cuda").manual_seed(F)
    theta = torch.randn(F, 22, 3, device="cuda", generator=gen) * 0.3
    tau = torch.randn(F, 3, device="cuda", generator=gen)
    init = theta + torch.randn(F, 22, 3, device="cuda", generator=gen) * 0.1
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")
    results = []
    for lay_name, lengths in layouts(F, 1).items():
        S = len(lengths)
        betas = torch.randn(S, 10, device="cuda", generator=gen)
        per_frame = torch.repeat_interleave(betas, torch.tensor(lengths, device="cuda"), dim=0)
        for name, model in (("mesh", mesh), ("synthetic", synth)):
            pack = model.keypoint_pack(torch.device("cuda"))
            nb = C.c_int64()
            L.check(L.lib().tik_fit_keypoints_shape_workspace_bytes(C.byref(pack.c), 17, 1, F, S, C.byref(nb)))
            nbytes = nb.value
            y = SU.keypoints(theta, model, per_frame, tau) + torch.randn(F, 17, 3, device="cuda", generator=gen) * 0.01
            for n_iter in [int(s) for s in args.iters.split(",")]:
                arms = {
                    "fit_keypoints_shape": lambda: SU.fit_keypoints_shape(y, model, init, lengths, None, tau, "coco", None,
                                                                          1e-3, 1e-3, n_iter),
                    "fit_keypoints": lambda: SU.fit_keypoints(y, model, init, None, tau, "coco", None, 1e-3, n_iter),
                }
                for run in arms.values():
                    for _ in range(args.warmup):
                        run()
                times = {k: [] for k in arms}
                outs = {}
                for _ in range(args.steps):
                    for k, run in arms.items():                      # alternate the two arms
                        flush.fill_(1.0)
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        outs[k] = run()
                        e1.record()
                        torch.cuda.synchronize()
                        times[k].append(e0.elapsed_time(e1) * 1e-3)
                t_s, t_k = float(np.median(times["fit_keypoints_shape"])), float(np.median(times["fit_keypoints"]))
                o = outs["fit_keypoints_shape"]
                r = {"layout": lay_name, "sequences": S, "model": name, "frames": F, "n_iter": n_iter,
                     "shape_ms": t_s * 1e3, "shape_ms_all": [x * 1e3 for x in times["fit_keypoints_shape"]],
                     "shape_M_frames_per_s": F / t_s / 1e6, "fit_keypoints_ms": t_k * 1e3,
                     "fit_keypoints_ms_all": [x * 1e3 for x in times["fit_keypoints"]],
                     "fit_keypoints_M_frames_per_s": F / t_k / 1e6, "ratio": t_s / t_k,
                     "launches": LAUNCHES_FIXED + LAUNCHES_PER_ITERATION * n_iter,
                     "launches_per_iteration": LAUNCHES_PER_ITERATION, "workspace_bytes_per_frame": nbytes / F,
                     "median_cost_ratio": float((o["cost"] / o["cost_init"]).median()),
                     "median_beta_error": float((o["betas"] - betas).abs().max(1).values.median())}
                results.append(r)
                print(f"{lay_name:>18} {name:>9} n_iter={n_iter:3d}: shape {t_s * 1e3:9.2f} ms ({F / t_s / 1e6:6.3f} M frames/s)"
                      f"  fit_keypoints {t_k * 1e3:9.2f} ms  ratio {t_s / t_k:5.2f}  ws {nbytes / F:.0f} B/frame"
                      f"  cost ratio {r['median_cost_ratio']:.2e}", flush=True)
            del y
    doc = {"tool": "tools/bench_fit_shape.py", **info, "steps": args.steps, "warmup": args.warmup, "select": "coco",
           "fit_transl": True, "prior_weight": 1e-3, "shape_prior_weight": 1e-3, "l2_flush_bytes": flush.numel() * 4,
           "results": results}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_fit_shape.json"), "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps({k: doc[k] for k in ("gpu", "power_limit", "max_sm_clock")}))


if __name__ == "__main__":
    main()
