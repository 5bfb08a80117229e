"""Body keypoint throughput: smpl_util.keypoints (one tik_body_keypoints launch, COCO-17 selection) at F = 1,048,576 and
8,388,608 on a V = 10,475 synthetic SmplxBodyModel and on a synthetic full-skeleton model, with shared and per-frame
betas; for comparison at F = 65,536 the routes that exist without it: lbs() + COCO gather and fk_body (60 joints) +
gather.  CUDA events per call, a 256 MB buffer overwritten between calls (L2 flushed).

    python tools/bench_keypoints.py --out DIR [--steps N] [--warmup W]

Bounds from the shapes, estimates: bytes per frame = pose (55 x 12) + per-frame betas (10 x 4) + transl (12) + 17 points
(204) against the project's measured copy peak (MEASURED_PEAKS.json hbm_gbs, else 6,534 GB/s); FMAs per frame = pose
blend (54 x 9 x 15) + shape blend (55 x 3 x 10 + 5 x 3 x 10) + Rodrigues and FK (~3.3 k) + skinning (~0.3 k) against
148 SMs x 128 FP32 lanes x the max SM clock.  The baseline routes are reported with the same per-frame figures so the
columns compare.  Writes DIR/bench_keypoints.json (DIR is created; nothing is written elsewhere)."""
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

FMA_POSE_BLEND = 54 * 9 * 15
FMA_SHAPE = 55 * 3 * 10 + 5 * 3 * 10
FMA_FK = 3300
FMA_SKIN = 300


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        name, power, clock = torch.cuda.get_device_name(0), "unknown", "unknown"
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def time_call(fn, flush, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) * 1e-3)
    return float(np.median(times)), float(min(times)), float(max(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for bench_keypoints.json")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--frames", default="1048576,8388608")
    ap.add_argument("--baseline-frames", type=int, default=65536)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_keypoints needs a GPU")
    info = gpu_info()
    hbm = 6534.1
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        hbm = json.load(open(p)).get("hbm_gbs", hbm)
    try:
        clock_ghz = float(info["max_sm_clock"].split()[0]) / 1000.0
    except (ValueError, IndexError):
        clock_ghz = 1.965
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    fma_peak = sms * 128 * clock_ghz * 1e9                       # FP32 FMAs per second
    V = 10475
    mesh = SU.SmplxBodyModel(smplx_synth.make_smplx_arrays(V, seed=0), skeleton="full")
    synth = SU.SyntheticBodyModel(skeleton="full")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    coco = SU.keypoint_indices("coco")
    results = []

    def record(route, model, F, betas_mode, t3, nbytes, fmas):
        t = t3[0]
        t_hbm, t_fma = F * nbytes / (hbm * 1e9), F * fmas / fma_peak
        r = {"route": route, "model": model, "frames": F, "betas": betas_mode, "median_s": t, "min_s": t3[1], "max_s": t3[2],
             "frames_per_s": F / t, "bytes_per_frame": nbytes, "achieved_gbs": F * nbytes / t / 1e9,
             "share_of_hbm_peak": t_hbm / t, "fma_per_frame": fmas, "share_of_fma_peak": t_fma / t,
             "bound": "fma" if t_fma >= t_hbm else "hbm", "share_of_bound": max(t_hbm, t_fma) / t}
        results.append(r)
        print(f"{route:>12} {model:>9} F={F:8d} betas={betas_mode:>6}: {t * 1e3:9.3f} ms  {F / t / 1e6:9.2f} M frames/s  "
              f"{r['achieved_gbs']:7.1f} GB/s  {r['share_of_bound'] * 100:5.1f} % of the {r['bound']} bound", flush=True)
        return r

    for F in [int(f) for f in args.frames.split(",")]:
        g = torch.Generator(device="cuda").manual_seed(F)
        pose = torch.randn(F, 55, 3, device="cuda", generator=g) * 0.4
        transl = torch.randn(F, 3, device="cuda", generator=g)
        per_frame = torch.randn(F, 10, device="cuda", generator=g)
        shared = np.linspace(-1, 1, 10)
        for name, model, blend in (("mesh", mesh, FMA_POSE_BLEND), ("synthetic", synth, 0)):
            for betas_mode, b in (("shared", shared), ("frame", per_frame)):
                t3 = time_call(lambda: SU.keypoints(pose, model, b, transl), flush, args.steps, args.warmup)
                nbytes = 55 * 12 + (40 if betas_mode == "frame" else 0) + 12 + 17 * 12
                record("keypoints", name, F, betas_mode, t3, nbytes, blend + FMA_SHAPE + FMA_FK + FMA_SKIN)
        del pose, transl, per_frame
        torch.cuda.empty_cache()

    F = args.baseline_frames
    g = torch.Generator(device="cuda").manual_seed(F)
    pose = torch.randn(F, 55, 3, device="cuda", generator=g) * 0.4
    transl = torch.randn(F, 3, device="cuda", generator=g)
    betas = np.linspace(-1, 1, 10)
    t3 = time_call(lambda: SU.lbs(pose, mesh, betas, transl)[0][:, coco], flush, args.steps, args.warmup)
    base_lbs = record("lbs+gather", "mesh", F, "shared", t3, 55 * 12 + 12 + 17 * 12,
                      FMA_POSE_BLEND + FMA_SHAPE + FMA_FK + FMA_SKIN)
    p60 = torch.cat([pose, torch.zeros(F, 5, 3, device="cuda")], 1)
    rest = synth.rest(betas)
    t3 = time_call(lambda: SU.fk_body(p60, rest, synth.parents, transl)[:, coco], flush, args.steps, args.warmup)
    base_fk = record("fk60+gather", "synthetic", F, "shared", t3, 55 * 12 + 12 + 17 * 12, FMA_FK)
    kp_mesh = max(r["frames_per_s"] for r in results if r["route"] == "keypoints" and r["model"] == "mesh" and r["betas"] == "shared")
    kp_syn = max(r["frames_per_s"] for r in results if r["route"] == "keypoints" and r["model"] == "synthetic" and r["betas"] == "shared")
    doc = {"tool": "tools/bench_keypoints.py", **info, "sms": sms, "hbm_peak_gbs": hbm, "fma_peak_per_s": fma_peak,
           "bounds_are_estimates": True, "steps": args.steps, "warmup": args.warmup, "l2_flushed": True, "results": results,
           "speedup_over_lbs_gather": kp_mesh / base_lbs["frames_per_s"],
           "speedup_over_fk60_gather": kp_syn / base_fk["frames_per_s"]}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_keypoints.json"), "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps({k: doc[k] for k in ("gpu", "power_limit", "max_sm_clock", "speedup_over_lbs_gather",
                                          "speedup_over_fk60_gather")}))


if __name__ == "__main__":
    main()
