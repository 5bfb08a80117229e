"""SMPL-X mesh skinning throughput: smpl_util.lbs (FK + pose features + pose-blend GEMM + skinning) at V = 10,475 on a
synthetic model (oracle/smplx_synth.py, same shapes as the licensed files), F = 16,384 (the poses of one configs[2] step)
and F = 65,536, fp32 and bf16, CUDA events per call with a 256 MB buffer overwritten between calls (L2 flushed).

    python tools/bench_mesh.py --out DIR [--steps N] [--warmup W] [--chunks auto,128,256,512,1024]

Bounds from the shapes: bytes = vertices written (F V 12) + poses read (F 55 12) + posedirs read once; FLOPs = pose blend
(2 F 486 3V) + skinning (F V (24 kmax + 18)).  HBM time against the project's measured copy peak (MEASURED_PEAKS.json
hbm_gbs, else 6,534 GB/s), GEMM time against its measured bf16 burst peak (1,576 TFLOP/s) for bf16 and a third of the
TF32 data-sheet rate (3 MMAs per product, 375 TFLOP/s) for fp32.  --chunks sweeps TIK_LBS_CHUNK (frames per chunk).
Writes DIR/bench_mesh.json (DIR is created; nothing is written elsewhere)."""
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


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        name, power, clock = torch.cuda.get_device_name(0), "unknown", "unknown"
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for bench_mesh.json")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--V", type=int, default=10475)
    ap.add_argument("--frames", default="16384,65536")
    ap.add_argument("--chunks", default="auto")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mesh needs a GPU")
    hbm = 6534.1
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        hbm = json.load(open(p)).get("hbm_gbs", hbm)
    gemm_peak = {"bf16": 1576e12, "fp32": 1125e12 / 3}
    V = args.V
    model = SU.SmplxBodyModel(smplx_synth.make_smplx_arrays(V, seed=0), skeleton="full",
                              landmark_vertex_ids=[i % V for i in SU.SMPLX_LANDMARK_VERTEX_IDS])
    rows = -(-3 * V // 128) * 128
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    betas = np.linspace(-1, 1, 10)
    results = []
    for F in [int(f) for f in args.frames.split(",")]:
        g = torch.Generator(device="cuda").manual_seed(F)
        pose = torch.randn(F, 55, 3, device="cuda", generator=g) * 0.4
        transl = torch.randn(F, 3, device="cuda", generator=g)
        for dtype in ("fp32", "bf16"):
            for chunk in args.chunks.split(","):
                if chunk == "auto":
                    os.environ.pop("TIK_LBS_CHUNK", None)
                else:
                    os.environ["TIK_LBS_CHUNK"] = chunk
                for _ in range(args.warmup):
                    SU.lbs(pose, model, betas, transl, dtype=dtype)
                torch.cuda.synchronize()
                times = []
                for _ in range(args.steps):
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    SU.lbs(pose, model, betas, transl, dtype=dtype)
                    e1.record()
                    torch.cuda.synchronize()
                    times.append(e0.elapsed_time(e1) * 1e-3)
                t = float(np.median(times))
                nbytes = F * V * 12 + F * 55 * 12 + rows * 512 * (2 if dtype == "bf16" else 4)
                flops_gemm = 2.0 * F * 486 * 3 * V
                flops = flops_gemm + F * V * (24.0 * model.kmax + 18)
                t_hbm, t_gemm = nbytes / (hbm * 1e9), flops_gemm / gemm_peak[dtype]
                bound = "hbm" if t_hbm >= t_gemm else "gemm"
                r = {"frames": F, "V": V, "dtype": dtype, "chunk": chunk, "kmax": model.kmax, "median_s": t,
                     "min_s": float(min(times)), "max_s": float(max(times)), "frames_per_s": F / t, "vertices_per_s": F * V / t,
                     "bytes": nbytes, "flops": flops, "achieved_gbs": nbytes / t / 1e9, "achieved_tflops": flops / t / 1e12,
                     "bound": bound, "bound_s": max(t_hbm, t_gemm), "share_of_bound": max(t_hbm, t_gemm) / t}
                results.append(r)
                print(f"F={F:6d} {dtype} chunk={chunk:>4}: {t * 1e3:8.3f} ms  {F / t / 1e6:6.2f} M frames/s  "
                      f"{F * V / t / 1e9:7.2f} G vertices/s  {nbytes / t / 1e9:7.1f} GB/s  {r['share_of_bound'] * 100:5.1f} % of the "
                      f"{bound} bound", flush=True)
    os.environ.pop("TIK_LBS_CHUNK", None)
    doc = {"tool": "tools/bench_mesh.py", **gpu_info(), "hbm_peak_gbs": hbm, "gemm_peak_flops": gemm_peak,
           "steps": args.steps, "warmup": args.warmup, "l2_flushed": True, "results": results}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_mesh.json"), "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps({k: doc[k] for k in ("gpu", "power_limit", "max_sm_clock")}))


if __name__ == "__main__":
    main()
