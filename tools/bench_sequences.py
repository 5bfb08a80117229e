"""Many sequences at once: inference.run_inference_batch against a loop of inference.run_inference.

Seeded synthetic COCO-17 keypoint sequences with log-uniform lengths in [60, 3000] frames, in batches of 1, 16, 256 and
2,048 sequences, under three configurations: the reference's default hparams (win 9, h_w_size 0) in fp32 and in bf16,
and win 65 with h_w_size 2 in rotation mode (bf16).  Two routes, each timed by the host clock from a list of numpy
arrays to a list of numpy arrays (copies and the final synchronisation included):
  loop   [run_inference(model, s, ...) for s in seqs]
  batch  run_inference_batch(model, seqs, ...)
and, separately, the device time of the batch route's GPU work (forward_windows(lengths=...) + window_mean(lengths=...)
on a resident packed buffer) by CUDA events.  Before timing, the two routes must agree: bit for bit in euclidean mode,
within 1e-6 in rotation mode.

    python tools/bench_sequences.py --out DIR [--steps N] [--warmup W] [--batches 1,16,256,2048]

Writes DIR/bench_sequences.json (DIR is created; nothing is written elsewhere)."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_keypoints import gpu_info  # noqa: E402
from oracle import stgcn_port as sp, synth  # noqa: E402
from temporal_inverse_kinematics_b200 import inference  # noqa: E402
from temporal_inverse_kinematics_b200.keypoints_util import COCO_ROOT_PAIR  # noqa: E402
from temporal_inverse_kinematics_b200.pose_regressor import IKPoseTrainer, default_hparams  # noqa: E402

CONFIGS = [("win9_h0_fp32", 9, 0, "euclidean", "fp32"), ("win9_h0_bf16", 9, 0, "euclidean", "bf16"),
           ("win65_h2_rotation_bf16", 65, 2, "rotation", "bf16")]


def make_sequences(n, seed):
    rs = np.random.RandomState(seed)
    lengths = np.exp(rs.uniform(np.log(60), np.log(3000), size=n)).astype(np.int64)
    return [(rs.standard_normal((int(F), 17, 3)) * 0.3).astype(np.float32) for F in lengths]


def host_time(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()                                  # ends in a device-to-host copy of the poses: synchronised
        times.append(time.perf_counter() - t0)
    return float(np.median(times)), float(min(times)), float(max(times))


def device_time(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) * 1e-3)
    return float(np.median(times)), float(min(times)), float(max(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for bench_sequences.json")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--batches", default="1,16,256,2048")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sequences needs a GPU")
    info = gpu_info()
    sd = synth.make_regressor_state(sp.build_adjacency("coco", "uniform", 2, 1), seed=0)
    results = []
    for name, win, h, mode, dtype in CONFIGS:
        tr = IKPoseTrainer(default_hparams(win_size=win)).eval()
        tr.regressor.load_state_dict(sd, strict=True)
        tr = tr.cuda()
        tr.regressor.set_compute_dtype(dtype)
        half = win // 2
        for S in [int(b) for b in args.batches.split(",")]:
            seqs = make_sequences(S, seed=1000 + S)
            lengths = [len(s) for s in seqs]
            frames = int(sum(lengths))
            loop = lambda: [inference.run_inference(tr, s, h_w_size=h, mean_mode=mode) for s in seqs]
            batch = lambda: inference.run_inference_batch(tr, seqs, h_w_size=h, mean_mode=mode)
            a, b = loop(), batch()
            for x, y in zip(a, b):
                if mode == "euclidean":
                    assert np.array_equal(x, y), f"{name} S={S}: routes differ"
                else:
                    assert np.abs(x - y).max() <= 1e-6, f"{name} S={S}: routes differ by {np.abs(x - y).max()}"
            del a, b
            t_loop = host_time(loop, args.steps, args.warmup)
            t_batch = host_time(batch, args.steps, args.warmup)
            packed = torch.from_numpy(np.concatenate(seqs)).cuda()

            def gpu_work():
                poses = tr.regressor.forward_windows(packed, 2 * half + 1, offset=-half, stride=1, root=COCO_ROOT_PAIR,
                                                     lengths=lengths)["poses"]
                return inference.window_mean(poses, h, mode, lengths=lengths)
            t_dev = device_time(gpu_work, args.steps, args.warmup)
            windows = frames                                   # one window per frame (offset = -win // 2)
            r = {"config": name, "win": win, "h_w_size": h, "mean_mode": mode, "dtype": dtype, "sequences": S,
                 "frames": frames, "windows": windows, "window_frames": windows * win,
                 "loop_s": t_loop[0], "loop_min_max_s": t_loop[1:], "batch_s": t_batch[0], "batch_min_max_s": t_batch[1:],
                 "device_s": t_dev[0], "device_min_max_s": t_dev[1:],
                 "loop_windows_per_s": windows / t_loop[0], "batch_windows_per_s": windows / t_batch[0],
                 "device_windows_per_s": windows / t_dev[0], "device_window_frames_per_s": windows * win / t_dev[0],
                 "loop_frames_per_s": frames / t_loop[0], "batch_frames_per_s": frames / t_batch[0],
                 "speedup": t_loop[0] / t_batch[0]}
            results.append(r)
            print(f"{name:>24} S={S:5d} frames={frames:8d}: loop {t_loop[0] * 1e3:9.2f} ms  batch {t_batch[0] * 1e3:9.2f} ms  "
                  f"x{r['speedup']:6.2f}  batch {r['batch_windows_per_s'] / 1e6:7.3f} M windows/s  device "
                  f"{t_dev[0] * 1e3:8.3f} ms = {r['device_windows_per_s'] / 1e6:7.3f} M windows/s "
                  f"({r['device_window_frames_per_s'] / 1e6:7.1f} M window-frames/s)", flush=True)
            del packed
            torch.cuda.empty_cache()
    doc = {"tool": "tools/bench_sequences.py", **info, "steps": args.steps, "warmup": args.warmup,
           "lengths": "log-uniform in [60, 3000], seeded", "timing": "host clock, list of numpy in -> list of numpy out; "
           "device_s: CUDA events around forward_windows(lengths) + window_mean(lengths)", "results": results}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_sequences.json"), "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps({k: doc[k] for k in ("gpu", "power_limit", "max_sm_clock")}))


if __name__ == "__main__":
    main()
