#!/usr/bin/env python
"""Benchmark of the learned-IK hot path: IK-solved frames/s (ST-GCN forward + SMPL-X body FK) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 0..4]

BASELINE.json configs (a "step" is one pass of the hot path over the config's synthetic workload):

  --config 2  (default, every N)  B=4096 clips/GPU, T=64, bf16 tensor-core ST-GCN forward + 22-joint body FK.
              With --gpus N each rank runs its own 4096 clips (weak scaling); the solved poses are all-gathered on a
              side stream that overlaps the next step.  The default run (no --config) appends a "configs3" block:
  --config 3  65,536 clips of T=128 (8.4 M frames) sharded contiguously over the N ranks, 2048-clip micro-batches,
              ONE NCCL all-gather of the poses at the end of the step (strong scaling).  Its 142 ms steps run under
              the power cap (~1.66 GHz) while configs[2]'s 4 ms steps run at 1.97 GHz, so the two are not mixed in
              one scaling series: the headline line is configs[2] at every N and carries configs[3] beside it.
  --config 1  B=256, T=64, fp32 (1e-4 parity path), both head variants (aa66 live head, rot6d132 iterative head +
              rot6d -> rotmat), 1 GPU.
  --config 4  one 8192-frame sequence, 64-frame windows, stride 1: bulk windows/s and batch-1 latency p50/p99.
  --config 0  the reference's own CPU case (dance_contemporary.npz, 231 windows of 9 frames, batch 1, fp32).

One process per GPU (torchrun for N>1); rank 0 prints ONE JSON line.  `value`: inputs resident in HBM, CUDA events
on the launching stream, L2 flushed between steps, max over ranks.  `e2e`: the same through the public API from
pinned host buffers, host<->device copies inside the timed region.  `parity`: max-abs / RMS of the GPU poses,
rotation matrices and FK joints against the CPU arm on the clips that arm computes (fails loudly above tolerance).

`--dump-outputs DIR` writes, after the timed steps, what the timed path computed in its last step as DIR/<name>.npy
(float32; rank 0's clips; a fixed, seeded sample of the clips when the arrays exceed 64 MB).  The inputs depend only on
the arguments, so two builds can be compared output for output.

`--impl reference` (and the `cpu_baseline` leg) time the reference's OWN PyTorch modules on the host cores when
oracle/_ref (snapshot made by oracle/build_ref.py) or /root/reference is present (kind "reference"), else the
oracle restatement (kind "port"); FK has no in-repo reference code (third-party smplx) and always uses the oracle's
numpy chain.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

V, C_IN, J = 17, 3, 22
METRIC = "IK-solved frames/sec (ST-GCN fwd + SMPL-X FK)"
UNIT = "frames/s"
CPU_SAMPLE_CLIPS = 256
CFG = {
    0: dict(name="configs[0]", T=9, dtype="fp32"),
    1: dict(name="configs[1]", B=256, T=64, dtype="fp32"),
    2: dict(name="configs[2]", B=4096, T=64, dtype="bf16"),
    3: dict(name="configs[3]", B=65536, T=128, dtype="bf16", micro=2048),
    4: dict(name="configs[4]", F=8192, T=64, dtype="bf16"),
}
# stated tolerances (max-abs, RMS) of the bf16 path on the quantities north_star gates; fp32: 1e-4 max-abs
TOL = {"bf16": {"poses": (0.08, 0.02), "rotmats": (0.08, 0.015), "joints": (0.08, 0.012)},
       "fp32": {"poses": (1e-4, 1e-4), "rotmats": (1e-4, 1e-4), "joints": (1e-4, 1e-4)}}

_JSON_OUT = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner there when NCCL_DEBUG is
    set) must not interleave with it: keep a private handle on the real stdout and point fd 1 at stderr."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def _emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes each array (clips along axis 0) as out_dir/<name>.npy in float32.  Above DUMP_LIMIT_BYTES in all, the
    same seeded sample of clips is taken from every array."""
    import numpy as np
    arrays = {k: np.ascontiguousarray(np.asarray(v, dtype=np.float32)) for k, v in arrays.items()}
    n = next(iter(arrays.values())).shape[0]
    assert all(a.shape[0] == n for a in arrays.values()), {k: a.shape for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        keep = max(1, n * DUMP_LIMIT_BYTES // total)
        idx = np.sort(np.random.RandomState(0).choice(n, keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


TC_KERNELS = ("rowgemm_umma", "rowgemm_ts", "tcn_halo", "gcn_fused", "gcn_wide", "stem_block", "block_fused")


def _ncu_traffic_per_launch():
    """dram__bytes_read.sum + dram__bytes_write.sum per tensor-core launch, averaged over one step of the newest
    committed ncu launch list under profiles/ (None if there is none)."""
    import csv
    import glob
    cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "r2_launches*.csv"))) or \
        sorted(glob.glob(os.path.join(ROOT, "profiles", "r1_launches_final.csv")))
    if not cands:
        return None, None
    p = cands[-1]
    per = {}
    with open(p) as f:
        rows = [r for r in csv.reader(l for l in f if l.startswith('"'))]
    if not rows:
        return None, None
    hdr = rows[0]
    ki, mi, vi, ii = hdr.index("Kernel Name"), hdr.index("Metric Name"), hdr.index("Metric Value"), hdr.index("ID")
    for r in rows[1:]:
        if any(k in r[ki] for k in TC_KERNELS) and r[mi].startswith("dram__bytes"):
            per[r[ii]] = per.get(r[ii], 0.0) + float(r[vi].replace(",", ""))
    return (sum(per.values()) / len(per) if per else None), os.path.relpath(p, ROOT)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 20 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index
        self.i0 = 0

    def mark(self):
        """Everything sampled from now on is inside the timed region (the process is started earlier: nvidia-smi
        needs tens of ms to produce its first row)."""
        self.i0 = len(self.rows)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        rows = self.rows[self.i0:] or self.rows
        sm = sorted(int(r[0]) for r in rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU / reference arm
class CpuArm:
    """The reference's CPU implementation of the path.  kind "reference": its own nn.Modules (pose_trainer.PoseRegressor
    from oracle/_ref or /root/reference, unmodified) carrying the synthetic state dict; kind "port": the oracle
    restatement.  FK (third-party smplx in the reference) is the oracle's numpy chain in both cases."""

    def __init__(self, want_port=False):
        import torch
        from oracle import fk_port, ref_import, stgcn_port as sp, synth
        self.torch, self.sp, self.synth, self.fk_port = torch, sp, synth, fk_port
        self.A = sp.build_adjacency("coco", "uniform", 2, 1)
        self.sd = synth.make_regressor_state(self.A, seed=0)
        self.rest, self.parents = synth.make_rest_skeleton(), synth.SMPLX_BODY_PARENTS
        self.kind, self.model, self.ref = "port", None, None
        if ref_import.available() and not want_port:
            self.ref = ref_import.load()
            self.model = self.ref.pose_trainer.PoseRegressor(ref_import.default_hparams()).eval()
            self.model.load_state_dict(self.sd, strict=True)
            self.kind = "reference"
            self.source = "oracle/_ref snapshot" if ref_import.is_snapshot() else ref_import.REF_ROOT

    def poses(self, x):
        with self.torch.no_grad():
            if self.model is not None:
                return self.model(x)["poses"]
            return self.sp.regressor_forward(self.sd, x)["poses"]

    def step(self, x):
        """PoseRegressor forward + FK of the solved poses -> (poses, local rotmats, joints) numpy."""
        import numpy as np
        poses = self.poses(x)
        aa = poses.reshape(-1, J, 3).numpy()
        joints, R, _ = self.fk_port.fk_from_axis_angle(aa.astype(np.float64), self.rest.astype(np.float64), self.parents)
        return poses.numpy(), R, joints

    def time(self, x, iters, warm=1, threads=None):
        torch = self.torch
        old = torch.get_num_threads()
        if threads:
            torch.set_num_threads(threads)
        try:
            for _ in range(warm):
                self.step(x)
            ts = []
            for _ in range(iters):
                t0 = time.perf_counter()
                out = self.step(x)
                ts.append(time.perf_counter() - t0)
        finally:
            used = torch.get_num_threads()
            torch.set_num_threads(old)
        sec = sum(ts) / len(ts)
        return x.shape[0] * x.shape[1] / sec, sec, used, out

    def describe(self):
        if self.kind == "reference":
            return f"the reference's own pose_trainer.PoseRegressor ({self.source}) + numpy FK chain (smplx is third-party)"
        return "oracle port of the reference PyTorch modules + numpy FK chain"


def dance_windows():
    """configs[0] input: dance_contemporary.npz -> moveai->COCO remap + axis swap (inference.py:121-133) ->
    InferenceDataset windows of 9 frames (data_amass.py:221-236).  The npz content travels inside tests/golden/dance.npz."""
    import numpy as np
    from oracle import stgcn_port as sp
    g = np.load(os.path.join(ROOT, "tests", "golden", "dance.npz"), allow_pickle=False)
    names = [str(s) for s in g["joint_3d_names"]]
    return sp.inference_windows(sp.moveai_to_coco(g["joints_3d"], names), 9).astype(np.float32), g["poses"]


def reference_workload(args, arm):
    """(x sample, description, frames-per-step, full-config flag) of the CPU arm for the chosen config."""
    import torch
    cfg = CFG[args.config]
    if args.config == 0:
        wins, _ = dance_windows()
        return torch.from_numpy(wins), "all 231 windows of 9 frames, batch 1 (the config verbatim)", True
    if args.config == 4:
        x = arm.synth.make_clips(32, cfg["T"], seed=100)
        return x, "32 windows of 64 frames, batch 1 (bounded sample of the 8129 windows)", False
    n = min(CPU_SAMPLE_CLIPS, cfg["B"])
    x = arm.synth.make_clips(n, cfg["T"], seed=1234)
    full = n == cfg["B"]
    return x, (f"{n} clips x T={cfg['T']} per step" + ("" if full else f" (bounded sample of the B={cfg['B']} clips)")), full


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    arm = CpuArm(want_port=args.port)
    cfg = CFG[args.config]
    x, sample, _ = reference_workload(args, arm)
    batch1 = args.config in (0, 4)
    steps, warm = max(1, args.steps), max(1, min(args.warmup, 2))

    def one_pass():
        if batch1:                                                # DataLoader(batch_size=1) loop of inference.py:43-52
            return [arm.step(x[i:i + 1]) for i in range(x.shape[0])]
        return [arm.step(x)]

    for _ in range(warm):
        one_pass()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        outs = one_pass()
        ts.append(time.perf_counter() - t0)
    if args.dump_outputs:
        import numpy as np
        poses = np.concatenate([o[0] for o in outs])
        joints = np.concatenate([o[2] for o in outs]).reshape(poses.shape[0], poses.shape[1], J, 3)
        dump_outputs(args.dump_outputs, {"poses": poses, "joints": joints})
    sec = sum(ts) / len(ts)
    fps = x.shape[0] * x.shape[1] / sec
    threads = torch.get_num_threads()
    sample = f"{sample}, fp32, torch CPU, {arm.describe()}"
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "strong" if args.config == 3 else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args.config, 1), "sample": sample},
            "cpu_baseline": {"value": fps, "unit": UNIT, "cores": threads, "kind": arm.kind, "sample": sample},
            "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if batch1:
        line["latency_us"] = {"per_window_mean": sec / x.shape[0] * 1e6}
    _emit(line)


def workload_name(config, world):
    c = CFG[config]
    if config == 0:
        return "configs[0]: dance_contemporary.npz, 231 windows of 9 frames, batch 1, fp32 ST-GCN forward (joint angles only)"
    if config == 1:
        return "configs[1]: B=256 clips, T=64, fp32 ST-GCN fwd (aa66 head) + rot6d132 head variant + rot6d->rotmat + 22-joint FK"
    if config == 2:
        return (f"configs[2]: B={c['B']} clips/GPU, T={c['T']}, bf16 ST-GCN fwd (PoseRegressor, random-init weights) + 22-joint "
                f"body FK on {c['B'] * c['T'] // 16} solved poses/GPU")
    if config == 3:
        return (f"configs[3]: {c['B']} clips, T={c['T']} (8.4 M frames), sharded over {world} GPU(s), {c['micro']}-clip "
                f"micro-batches, bf16 ST-GCN fwd + 22-joint FK, ONE all-gather of the poses at the end")
    return "configs[4]: one 8192-frame sequence, windows of 64 frames, stride 1 (8129 windows), bf16, windows gathered in-kernel"


# ------------------------------------------------------------------------------------------------ our arm
def _parity(name_dtype, got, want):
    """got / want: dicts poses / rotmats / joints (numpy).  Returns the block, raises above the stated tolerance."""
    import numpy as np
    block, bad = {}, []
    for k in ("poses", "rotmats", "joints"):
        e = np.abs(np.asarray(got[k], dtype=np.float64) - np.asarray(want[k], dtype=np.float64))
        mx, rms = float(e.max()), float(np.sqrt((e ** 2).mean()))
        tol = TOL[name_dtype][k]
        block[k] = {"max_abs": mx, "rms": rms, "tol_max_abs": tol[0], "tol_rms": tol[1]}
        if not (mx < tol[0] and rms < tol[1]):
            bad.append(f"{k}: max-abs {mx:.3g} rms {rms:.3g} (tolerance {tol[0]} / {tol[1]})")
    block["ok"] = not bad
    if bad:
        raise SystemExit("bench.py: GPU result differs from the CPU arm beyond the stated tolerance: " + "; ".join(bad))
    return block


def _hbm_rooflines(dev, peaks, frames):
    """Stand-alone launches of the HBM-bound kernels at `frames` frames x 22 joints (SURVEY.md 8d): algorithmic bytes
    per frame / CUDA-event time, L2 flushed before each launch."""
    import torch
    from temporal_inverse_kinematics_b200 import geometry as G, kornia_geometry_conversion as KG, smpl_util as SU, synthetic
    M = frames * J
    g = torch.Generator(device=dev).manual_seed(5)
    x6 = torch.randn(M, 6, device=dev, generator=g)
    aa = torch.randn(M, 3, device=dev, generator=g) * 0.7
    R = G.batch_rodrigues(aa).view(-1, 3, 3)
    rest, parents = synthetic.make_rest_skeleton(), synthetic.SMPLX_BODY_PARENTS
    pose = aa.view(frames, J, 3)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {}
    cases = [("rot6d_to_rotmat", lambda: G.rot6d_to_rotmat(x6), 22 * 60),
             ("angle_axis_to_rotation_matrix", lambda: KG.angle_axis_to_rotation_matrix(aa), 22 * 48),
             ("batch_rodrigues", lambda: G.batch_rodrigues(aa), 22 * 48),
             ("rotation_matrix_to_angle_axis", lambda: G.rotation_matrix_to_angle_axis(R), 22 * 48),
             ("fk_body_joints", lambda: SU.fk_body(pose, rest, parents), 528),
             ("fk_body_joints_local_R", lambda: SU.fk_body(pose, rest, parents, want_local=True), 1320)]
    for name, fn, bpf in cases:
        for _ in range(2):
            fn()
        torch.cuda.synchronize(dev)
        tot, reps = 0.0, 5
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            tot += e0.elapsed_time(e1)
        sec = tot / reps * 1e-3
        gbs = frames * bpf / sec / 1e9
        out[name] = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                     "bytes_per_frame": bpf, "ms": sec * 1e3, "frames_per_s": frames / sec}
    del x6, aa, R, pose
    m = SU.SyntheticBodyModel("neutral", skeleton="full")
    f2 = frames // 4
    pose60 = torch.randn(f2, 60, 3, device=dev, generator=g) * 0.5
    for _ in range(2):
        SU.fk_body(pose60, m.rest_joints, m.parents)
    torch.cuda.synchronize(dev)
    tot = 0.0
    for _ in range(5):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        SU.fk_body(pose60, m.rest_joints, m.parents)
        e1.record()
        e1.synchronize()
        tot += e0.elapsed_time(e1)
    sec = tot / 5 * 1e-3
    gbs = f2 * 1440 / sec / 1e9
    out["fk_full_skeleton_60"] = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                                  "bytes_per_frame": 1440, "ms": sec * 1e3, "frames_per_s": f2 / sec, "frames": f2}
    return out


def pin_to_gpu_numa_node(local):
    """Bind this rank's threads to the CPUs nearest its GPU (NVML's ideal affinity), BEFORE any pinned host memory is
    allocated: the e2e leg moves 62 MB per 4 ms step per GPU through host memory, and with 8 ranks on a two-socket host
    half of them otherwise stage their copies on the far socket.  Best effort: returns the number of CPUs bound, or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        return None


def run_ours(args):
    import copy
    import torch
    import torch.distributed as dist
    from temporal_inverse_kinematics_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    args.numa_cpus = pin_to_gpu_numa_node(local) if world > 1 else None     # one rank: leave every host thread to the CPU arm
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.check(_lib.lib().tik_check_device())
    cfg = CFG[args.config]
    dtype = args.dtype or cfg["dtype"]
    if args.config in (0, 4):
        if world > 1:
            raise SystemExit(f"--config {args.config} is a single-GPU configuration")
        return run_ours_windows(args, dev, dtype)
    line = measure(args, dev, world, rank, local)
    if args.config == 2 and args.with_c3:
        # the stated multi-GPU workload (configs[3]: 65,536 clips of T=128 sharded over the ranks, ONE gather) in the same
        # run, so that every N of a scaling series carries it next to the configs[2] headline
        a3 = copy.copy(args)
        a3.config, a3.steps, a3.warmup, a3.no_cpu, a3.no_hbm, a3.batch, a3.dtype = 3, min(args.steps, 5), 3, True, True, 0, None
        a3.dump_outputs = None                                   # --dump-outputs writes the headline configs[2] results
        l3 = measure(a3, dev, world, rank, local)
        if rank == 0:
            line["configs3"] = {k: l3[k] for k in ("value", "unit", "ms_per_step", "scaling", "e2e", "clocks", "steps", "warmup") if k in l3}
            line["configs3"]["workload"] = l3["config"]["workload"]
            line["configs3"]["gather"] = l3["config"]["gather"]
            line["configs3"]["ranks"] = l3.get("ranks")
            line["configs3"]["note"] = ("sustained: 8.4 M frames per step keep the GPU under its power cap (lower SM clocks than the "
                                        "4 ms configs[2] steps separated by L2 flushes); compare configs3 values across N with each other")
    if rank == 0:
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


def measure(args, dev, world, rank, local):
    """One configs[1..3] measurement; returns the JSON line on rank 0 (None elsewhere)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from temporal_inverse_kinematics_b200 import smpl_util, synthetic as synth
    from temporal_inverse_kinematics_b200.distributed import shard_bounds
    from temporal_inverse_kinematics_b200.graph import Graph
    from temporal_inverse_kinematics_b200.pose_regressor import IterativePoseRegressor, PoseRegressor, default_hparams
    cfg = CFG[args.config]
    dtype = args.dtype or cfg["dtype"]

    T = cfg["T"]
    A = Graph("coco", "uniform", 2, 1).A
    model = PoseRegressor(default_hparams()).eval()
    model.load_state_dict(synth.make_regressor_state(A, seed=0))
    model = model.to(dev).set_compute_dtype(dtype)
    if args.chunk:
        model.chunk_clips = args.chunk
    model.use_cuda_graph = not args.no_graph
    rest, parents = synth.make_rest_skeleton(), synth.SMPLX_BODY_PARENTS
    T_out = model.backbone.out_frames(T)

    # ---- the rank's clips: [lo, hi) of the job, processed in micro-batches of `micro` clips
    if args.config == 3:
        total = args.batch or cfg["B"]
        lo, hi = shard_bounds(total, rank, world)
        micro = min(cfg["micro"], hi - lo)
        scaling = "strong"
    else:
        per_gpu = args.batch or cfg["B"]
        total, lo, hi, micro, scaling = world * per_gpu, rank * per_gpu, (rank + 1) * per_gpu, per_gpu, "weak"
    n_local = hi - lo
    n_sample = min(CPU_SAMPLE_CLIPS, n_local)
    x_host = torch.empty((n_local, T, V, C_IN), dtype=torch.float32).pin_memory()
    gen = torch.Generator(device=dev).manual_seed(99 + rank)
    for m0 in range(0, n_local, micro):                          # synthetic root-relative clips, generated on the device
        m1 = min(n_local, m0 + micro)
        xm = torch.randn((m1 - m0, T, V, C_IN), device=dev, generator=gen) * 0.3
        xm = xm - 0.5 * (xm[:, :, 11] + xm[:, :, 12])[:, :, None, :]
        x_host[m0:m1].copy_(xm)
    if rank == 0:                                                # the clips the CPU arm also solves (same seed)
        x_host[:n_sample].copy_(synth.make_clips(n_sample, T, seed=1234))
    x_dev = x_host.to(dev)
    poses_local = torch.empty((n_local, T_out, 66), device=dev)
    joints_local = torch.empty((n_local * T_out, J, 3), device=dev)
    mbs = [(m0, min(n_local, m0 + micro)) for m0 in range(0, n_local, micro)]
    sizes = [shard_bounds(total, r, world)[1] - shard_bounds(total, r, world)[0] for r in range(world)] if args.config == 3 else [n_local] * world
    assert len(set(sizes)) == 1 or world == 1, "bench shards are equal-sized (65,536 and 4096*N divide by 1/2/4/8)"
    RING = 4                                                     # configs[2] at N>1: steps a rank may run ahead of its gathers
    n_gath = 2 if args.config == 3 else RING
    gathered = [torch.empty((world * n_local, T_out, 66), device=dev) for _ in range(n_gath)] if world > 1 else None
    snaps = [torch.empty_like(poses_local) for _ in range(RING)] if (world > 1 and args.config != 3) else None
    snap_ready = [torch.cuda.Event() for _ in range(RING)]
    snap_free = [torch.cuda.Event() for _ in range(RING)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    main_stream = torch.cuda.current_stream(dev)
    side = torch.cuda.Stream(device=dev)
    gather_ms = []
    for e in snap_free:
        e.record(main_stream)

    # a second set of result buffers for the end-to-end loop: step i+1 computes into one while step i's D2H reads the other
    poses_bufs = [poses_local, torch.empty_like(poses_local)]
    joints_bufs = [joints_local, torch.empty_like(joints_local)]

    def solve(xm, m0, m1, b=0):
        poses = model(xm)["poses"]                               # (n, T', 66) axis-angle
        poses_bufs[b][m0:m1].copy_(poses)
        joints_bufs[b][m0 * T_out:m1 * T_out].copy_(smpl_util.fk_body(poses.view(-1, J, 3), rest, parents))

    def gather(i, timed=False, b=0):
        """configs[3]: ONE all-gather per step, on the compute stream (it ends the job).  configs[2] at N>1: the
        gather of step i runs on a side stream and overlaps step i+1 (double-buffered destination)."""
        if world == 1:
            return
        if args.config == 3:
            if timed:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                gather_ms.append((e0, e1))
                e0.record(main_stream)
            dist.all_gather_into_tensor(gathered[i % 2], poses_bufs[b])
            if timed:
                e1.record(main_stream)
        else:
            # The step's poses are snapshotted on the compute stream (4 MB device copy) into a ring of RING buffers; the
            # side stream gathers them.  A rank only waits for its own gather of RING steps ago, so the ranks are not
            # locked to the slowest GPU of every single step (power-cap jitter), only to the slowest GPU over the run.
            k = i % RING
            main_stream.wait_event(snap_free[k])
            snaps[k].copy_(poses_bufs[b])
            snap_ready[k].record(main_stream)
            with torch.cuda.stream(side):
                side.wait_event(snap_ready[k])
                dist.all_gather_into_tensor(gathered[k], snaps[k])
                snap_free[k].record(side)

    def step(x, i=0, timed=False):
        for m0, m1 in mbs:
            solve(x[m0:m1], m0, m1)
        gather(i, timed)                                         # (device-resident loops use result buffer 0)

    def barrier():
        main_stream.wait_stream(side)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                                          # running before the warm-up; rows are kept from mark() on
    for i in range(max(args.warmup, 3)):
        step(x_dev, i)
    barrier()

    # ---- device-resident timing: CUDA events per step on the launching stream, L2 flushed between steps
    sampler.mark()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for i, (a, b) in enumerate(ev):
        flush.zero_()
        a.record()
        step(x_dev, i, timed=True)
        b.record()
    t_end = torch.cuda.Event(enable_timing=True)
    main_stream.wait_stream(side)                                # the last overlapped gather belongs to the timed region
    t_end.record()
    barrier()
    ms_steps = sorted(a.elapsed_time(b) for a, b in ev)
    ms = (sum(ms_steps) + max(0.0, ev[-1][1].elapsed_time(t_end))) / args.steps
    g_ms = sum(a.elapsed_time(b) for a, b in gather_ms) / len(gather_ms) if gather_ms else 0.0
    # the end-to-end loop below computes into the same buffers: keep the last timed step's results as they are now
    last_step = {"poses": poses_local.cpu(), "joints": joints_local.view(n_local, T_out, J, 3).cpu()} \
        if (rank == 0 and args.dump_outputs) else None

    # ---- end to end through the public API: pinned host input -> H2D -> forward + FK -> (gather) -> D2H of the results
    # The copies are pipelined the way a serving loop would: the H2D copy of micro-batch k+1 runs on a copy stream
    # while micro-batch k computes (two device input buffers); the D2H read-back of step i overlaps step i+1.
    out_p = torch.empty((world * n_local if (rank == 0 and args.config == 3) else n_local, T_out, 66), dtype=torch.float32).pin_memory()
    out_j = torch.empty((n_local * T_out, J, 3), dtype=torch.float32).pin_memory()
    copy_stream = torch.cuda.Stream(device=dev)
    x_bufs = [torch.empty((micro, T, V, C_IN), device=dev) for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    done = torch.cuda.Event()
    read_back = [torch.cuda.Event(), torch.cuda.Event()]        # per result buffer: its D2H copies have finished

    def upload(k):
        m0, m1 = mbs[k % len(mbs)]
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[k % 2])              # the buffer's previous reader has finished
            x_bufs[k % 2][:m1 - m0].copy_(x_host[m0:m1], non_blocking=True)
            ready[k % 2].record(copy_stream)

    def e2e_run(n_steps):
        for e in consumed:
            e.record(main_stream)
        for e in read_back:
            e.record(copy_stream)
        k, n_mb = 0, len(mbs)
        upload(0)
        for i in range(n_steps):
            b = i % 2
            main_stream.wait_event(read_back[b])                 # step i-2's results have left this result buffer
            for m0, m1 in mbs:
                main_stream.wait_event(ready[k % 2])
                solve(x_bufs[k % 2][:m1 - m0], m0, m1, b)
                consumed[k % 2].record(main_stream)
                if k + 1 < n_steps * n_mb:
                    upload(k + 1)
                k += 1
            gather(i, b=b)
            if world > 1 and args.config != 3:
                main_stream.wait_stream(side)
            done.record(main_stream)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(done)
                src_p = gathered[i % 2] if (world > 1 and rank == 0 and args.config == 3) else poses_bufs[b]
                out_p.copy_(src_p, non_blocking=True)
                out_j.copy_(joints_bufs[b], non_blocking=True)
                read_back[b].record(copy_stream)
        main_stream.wait_stream(copy_stream)

    e2e_run(2)                                                   # warm-up of the pipelined loop (pinned buffers, copy stream)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    e2e_run(args.steps)
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1) / args.steps
    clocks = sampler.stop() if rank == 0 else None

    # ---- parity of what the last step computed, against the CPU arm on the same clips (rank 0).  After the timed
    # regions: seconds of CPU-only work just before them would let the GPU fall into an idle power state.
    parity = cpu = None
    if rank == 0 and not args.no_cpu:
        torch.set_num_threads(os.cpu_count() or 1)
        arm = CpuArm(want_port=args.port)
        xs = x_host[:n_sample].clone()
        fps, sec, threads, (w_poses, w_R, w_joints) = arm.time(xs, 3)
        pg = poses_local[:n_sample]
        jg, Rg = smpl_util.fk_body(pg.reshape(-1, J, 3), rest, parents, want_local=True)
        # joints: what the timed step itself produced (joints-only FK kernel); rotmats: the local rotations of the
        # same poses from the FK kernel's want_local variant
        got = {"poses": pg.cpu().numpy(), "rotmats": Rg.cpu().numpy(), "joints": joints_local[:n_sample * T_out].cpu().numpy()}
        del jg
        parity = _parity(dtype, got, {"poses": w_poses, "rotmats": w_R, "joints": w_joints})
        parity["clips"] = n_sample
        parity["against"] = arm.kind
        n1 = max(8, n_sample // 8)
        fps1, sec1, _, _ = arm.time(xs[:n1], 1, warm=0, threads=1)
        cpu = {"value": fps, "unit": UNIT, "cores": threads, "kind": arm.kind,
               "sample": f"{n_sample} of the {n_local} clips (T={T}), 3 iterations, {arm.describe()}; {sec:.2f} s/iteration",
               "one_thread": {"value": fps1, "clips": n1, "s_per_iteration": sec1}, "host_cpus": os.cpu_count()}

    t = torch.tensor([ms, ms_e2e, g_ms], device=dev, dtype=torch.float64)
    t_min = t.clone()
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(t_min, op=dist.ReduceOp.MIN)
    ms_own = ms
    ms, ms_e2e, g_ms = float(t[0]), float(t[1]), float(t[2])

    if rank == 0:
        peaks, peak_src = _peaks()
        frames = total * T
        plan = model.plan_for(micro, T)
        kinds, gemm_flops = plan.profile(x_dev[:micro])          # CUDA events around every kernel (one extra run)
        k_ms, k_n = kinds["gemm"]
        achieved = gemm_flops / (k_ms * 1e-3) / 1e12 if k_ms > 0 else 0.0
        if dtype == "bf16":
            peak, peak_name = peaks["bf16_tflops"], f"{peak_src} bf16_tflops (burst: cuBLAS 8192^3, best of 10)"
            kern = "tcgen05 family: rowgemm_umma_kernel / rowgemm_ts_kernel / tcn_halo_kernel / gcn_fused_kernel / gcn_wide_kernel / stem_block_kernel"
        else:
            if os.environ.get("TIK_NO_TF32"):
                peak, peak_name = 74.0, "nominal fp32 SIMT: 148 SM x 128 FMA x 2 x 1.965 GHz"
                kern = "rowgemm_f32_kernel"
            else:
                peak, peak_name = 1125.0 / 3.0, "nominal dense TF32 1125 TFLOP/s (B200_PROFILING.md) / 3 MMAs per fp32 product (3xTF32 split)"
                kern = "rowgemm_tf32_kernel (tcgen05.mma kind::tf32, 3xTF32, per-chunk accumulation)"
        traffic, traffic_src = _ncu_traffic_per_launch()
        launches_per_step = len(mbs) * (plan.launches(micro) + 1)   # + FK per micro-batch
        roofline = {"bound": "tensor", "kernel": kern, "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                    "frac": achieved / peak, "peak_source": peak_name, "launches": k_n,
                    "avg_launch_us": k_ms * 1e3 / max(k_n, 1), "flops_per_launch_set": gemm_flops,
                    "kernel_ms_per_micro_batch": {k: v[0] for k, v in kinds.items()},
                    "traffic": traffic if dtype == "bf16" else None, "traffic_source": traffic_src if dtype == "bf16" else None,
                    "whole_step": {"achieved": frames / world * 7.991e6 / (ms * 1e-3) / 1e12, "unit": "TFLOP/s",
                                   "frac": frames / world * 7.991e6 / (ms * 1e-3) / 1e12 / peak,
                                   "note": "7.991 MFLOP per input frame (SURVEY 8d) x frames per GPU / step time"}}
        if dtype == "bf16":
            roofline["frac_of_sustained_peak"] = achieved / peaks["bf16_tflops_sustained"]
            if traffic and k_ms > 0:
                gbs = traffic / (roofline["avg_launch_us"] * 1e-6) / 1e9
                roofline["dram"] = {"achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                                    "note": "DRAM bytes per launch from the committed ncu capture / live launch time"}
        line = {"metric": METRIC, "value": frames / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms, "ms_per_step_min_median_max_rank0": [ms_steps[0], ms_steps[len(ms_steps) // 2], ms_steps[-1]],
                "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
                "dtype": dtype, "data": "synthetic",
                "config": {"workload": workload_name(args.config, world), "global_batch": total, "clips_per_gpu": n_local,
                           "frames_per_step": frames, "micro_batch_clips": micro, "chunk_clips": plan.n_chunk,
                           "cuda_graph": bool(model.use_cuda_graph), "l2": "flushed between timed steps (256 MiB memset)",
                           "parallelism": f"dp{world}",
                           "gather": ("none" if world == 1 else "ONE NCCL all_gather of the poses at the end of the step, on the compute stream"
                                      if args.config == 3 else "NCCL all_gather of the poses per step on a side stream from a 4-deep snapshot ring (overlaps the next steps)"),
                           "e2e_pipeline": "pinned H2D of micro-batch k+1 and D2H of step i's results (double-buffered) overlap compute on a copy stream",
                           "host_affinity": (f"rank 0 bound to the {args.numa_cpus} CPUs NVML names nearest its GPU" if getattr(args, "numa_cpus", None)
                                             else "unbound")},
                "e2e": {"value": frames / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                        "note": "every step: pinned-host input -> H2D -> model(x) + fk_body -> D2H of poses and joints, all inside the timed "
                                "region, copies overlapped on a copy stream; no L2 flush here (the step's input arrives over PCIe), "
                                "which is why it can match the flushed device-resident number",
                        "h2d_bytes_per_step": world * x_host.numel() * 4,
                        "d2h_bytes_per_step": (out_p.numel() + world * out_j.numel() + (0 if args.config == 3 else (world - 1) * out_p.numel())) * 4},
                "gpu_launches": launches_per_step * args.steps, "clocks": clocks, "roofline": roofline,
                "clips_per_s": total / (ms * 1e-3), "output_poses_per_s": total * T_out / (ms * 1e-3)}
        if world > 1:
            line["ranks"] = {"ms_per_step_max": ms, "ms_per_step_min": float(t_min[0]), "ms_per_step_rank0": ms_own,
                             "gather_ms_per_step": g_ms if args.config == 3 else None,
                             "gather_bytes_per_rank": poses_local.numel() * 4}
        if parity is not None:
            line["parity"] = parity
        if cpu is not None and world == 1:
            line["cpu_baseline"] = cpu
        if world == 1 and args.config == 2 and not args.no_hbm:
            line["roofline_hbm"] = _hbm_rooflines(dev, peaks, args.hbm_frames)
        if args.config == 1:
            line["rot6d132_head"] = _config1_rot6d(dev, IterativePoseRegressor, default_hparams, synth, A, x_dev, args)
        if last_step is not None:
            dump_outputs(args.dump_outputs, {k: v.numpy() for k, v in last_step.items()})
        return line
    return None


def _config1_rot6d(dev, IterativePoseRegressor, default_hparams, synth, A, x_dev, args):
    """configs[1]'s second head variant: iterative 6-D head + rot6d -> rotmat (+ rotmat -> axis-angle), fp32."""
    import torch
    m = IterativePoseRegressor(default_hparams()).eval()
    m.load_state_dict(synth.make_iterative_state(A, seed=0))
    m = m.to(dev).set_compute_dtype("fp32")
    for _ in range(30):                                          # also brings the clocks back up after the CPU arm
        m(x_dev)
    torch.cuda.synchronize(dev)
    times = []
    for _ in range(max(args.steps, 10)):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = m(x_dev)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = sorted(times)[len(times) // 2]                          # median: single steps occasionally catch a clock ramp
    R = out["rotmats"].reshape(-1, 3, 3)
    ortho = float((R @ R.transpose(1, 2) - torch.eye(3, device=dev)).abs().max())
    return {"ms_per_step": ms, "frames_per_s": x_dev.shape[0] * x_dev.shape[1] / (ms * 1e-3), "rotmats": list(out["rotmats"].shape),
            "max_orthonormality_error": ortho}


def run_ours_windows(args, dev, dtype):
    """configs[0] (231 windows of 9 frames, batch 1) and configs[4] (8192-frame sequence, 64-frame windows)."""
    import numpy as np
    import torch
    from temporal_inverse_kinematics_b200 import synthetic as synth
    from temporal_inverse_kinematics_b200.graph import Graph
    from temporal_inverse_kinematics_b200.pose_regressor import PoseRegressor, default_hparams
    cfg = CFG[args.config]
    model = PoseRegressor(default_hparams()).eval()
    model.load_state_dict(synth.make_regressor_state(Graph("coco", "uniform", 2, 1).A, seed=0))
    model = model.to(dev).set_compute_dtype(dtype)
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    W = cfg["T"]
    parity = None
    if args.config == 0:
        wins, golden_poses = dance_windows()
        xs = [torch.from_numpy(wins[i:i + 1]).to(dev) for i in range(wins.shape[0])]
        x_host = torch.from_numpy(wins).pin_memory()
        got = torch.cat([model(x)["poses"] for x in xs]).cpu().numpy()
        err = float(np.abs(got - golden_poses).max())              # tests/golden/dance.npz: the real reference's output
        if dtype == "fp32" and err > 1e-4:
            raise SystemExit(f"bench.py: configs[0] poses differ from the reference golden by {err}")
        parity = {"poses": {"max_abs": err, "tol_max_abs": 1e-4 if dtype == "fp32" else 0.08}, "against": "reference golden (tests/golden/dance.npz)",
                  "ok": True, "clips": len(xs)}
        bulk_fn = lambda: model(x_host.to(dev, non_blocking=True))["poses"]
        n_bulk = len(xs)
    else:
        seq = synth.make_clips(1, cfg["F"], seed=5)[0].to(dev)
        n_bulk = cfg["F"] - W + 1
        xs = [synth.make_clips(1, W, seed=100 + i).to(dev) for i in range(8)]
        bulk_fn = lambda: model.forward_windows(seq, W, offset=0, stride=1, root=(11, 12))["poses"]
    for _ in range(max(args.warmup, 3)):
        bulk_fn()
    torch.cuda.synchronize(dev)
    sampler.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        y_bulk = bulk_fn()
    e1.record()
    e1.synchronize()
    ms_bulk = e0.elapsed_time(e1) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"poses": y_bulk.cpu().numpy()})
    # batch 1 through the public API: device latency (events) and host-observed latency incl. D2H, (a) on the
    # throughput plan with CUDA-graph replay (19-25 launches), (b) on the latency plan (one persistent cooperative
    # kernel, fp32) -- the one a streaming caller selects with model.low_latency = True
    out_host = torch.empty((1, model.backbone.out_frames(W), 66)).pin_memory()
    n_lat = 2000 if args.config == 4 else len(xs) * 4
    q = lambda a, p: float(np.percentile(np.array(a), p))

    def latency_run(fn=None):
        call = fn or (lambda x: model(x)["poses"])
        for x in xs[:8]:
            call(x)
        torch.cuda.synchronize(dev)
        dev_us, host_us = [], []
        for i in range(n_lat):
            x = xs[i % len(xs)]
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            a.record()
            y = call(x)
            b.record()
            out_host.copy_(y, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
            host_us.append((time.perf_counter() - t0) * 1e6)
            dev_us.append(a.elapsed_time(b) * 1e3)
        return dev_us, host_us, y

    model.use_cuda_graph = True
    g_dev, g_host, y_graph = latency_run()
    graph_plan = model.plan_for(1, W)
    model.low_latency = True
    dev_us, host_us, y_lat = latency_run()
    s_dev, s_host, y_ses = latency_run(model.session(1, W))      # bound forward: plan resolved once, launch only
    assert torch.equal(y_ses, y_lat)
    clocks = sampler.stop()
    plan = model.plan_for(1, W)
    lat_vs_graph = float((y_lat - y_graph).abs().max())
    line = {"metric": METRIC, "value": n_bulk * W / (ms_bulk * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_bulk, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": dtype, "data": "synthetic" if args.config == 4 else "dance_contemporary.npz (via tests/golden/dance.npz), random-init weights",
            "config": {"workload": workload_name(args.config, 1), "windows": n_bulk, "window_frames": W,
                       "value_is": "all windows in one pass (window-frames/s); batch-1 latency in latency_us",
                       "cuda_graph": True},
            "windows_per_s": n_bulk / (ms_bulk * 1e-3),
            "latency_us": {"steps": n_lat, "plan": "latency plan: one persistent cooperative kernel, fp32 (model.low_latency)",
                           "device_p50": q(dev_us, 50), "device_p99": q(dev_us, 99),
                           "host_incl_d2h_p50": q(host_us, 50), "host_incl_d2h_p99": q(host_us, 99),
                           "launches_per_window": plan.launches(1), "phases": getattr(plan, "phases", None),
                           "max_abs_vs_throughput_plan": lat_vs_graph,
                           "session": {"what": "model.session(1, T): plan resolved once, per-call work = allocate the output + one launch",
                                       "device_p50": q(s_dev, 50), "device_p99": q(s_dev, 99),
                                       "host_incl_d2h_p50": q(s_host, 50), "host_incl_d2h_p99": q(s_host, 99)},
                           "throughput_plan_cuda_graph": {"device_p50": q(g_dev, 50), "device_p99": q(g_dev, 99),
                                                          "host_incl_d2h_p50": q(g_host, 50), "host_incl_d2h_p99": q(g_host, 99),
                                                          "launches_per_window": graph_plan.launches(1), "dtype": dtype}},
            "e2e": {"value": W * 1e6 / q(host_us, 50), "unit": UNIT, "note": "batch 1: frames of one window / host-observed p50 latency incl. D2H",
                    "h2d_bytes_per_step": 0 if args.config == 4 else W * V * C_IN * 4, "d2h_bytes_per_step": out_host.numel() * 4},
            "gpu_launches": plan.launches(1) * n_lat, "clocks": clocks}
    if parity:
        line["parity"] = parity
    if not args.no_cpu:
        torch.set_num_threads(os.cpu_count() or 1)
        arm = CpuArm(want_port=args.port)
        xs_cpu = [x.cpu() for x in xs[:32]]
        t0 = time.perf_counter()
        for x in xs_cpu:
            arm.poses(x)
        sec = (time.perf_counter() - t0) / len(xs_cpu)
        line["cpu_baseline"] = {"value": W / sec, "unit": UNIT, "cores": torch.get_num_threads(), "kind": arm.kind,
                                "sample": f"{len(xs_cpu)} windows of {W} frames, batch 1, {arm.describe()} (no FK); {sec * 1e3:.1f} ms/window"}
    _emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=None, choices=sorted(CFG),
                    help="BASELINE.json configs index (default: 2 = B=4096 clips/GPU, T=64, at every N, plus a configs[3] block)")
    ap.add_argument("--no-c3", action="store_true", help="default run only: skip the additional configs[3] block")
    ap.add_argument("--dtype", default=None, choices=["bf16", "fp32"], help="override the config's compute dtype")
    ap.add_argument("--batch", type=int, default=0, help="clips per GPU (config 2) / total clips (config 3)")
    ap.add_argument("--chunk", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU arm (no cpu_baseline, no parity block)")
    ap.add_argument("--no-hbm", action="store_true", help="skip the stand-alone HBM-kernel rooflines")
    ap.add_argument("--hbm-frames", type=int, default=1 << 23)
    ap.add_argument("--port", action="store_true", help="CPU arm: use the oracle restatement even if the reference modules are present")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels one by one instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's results (poses, joints) as DIR/<name>.npy, float32, 64 MB at most")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    args.with_c3 = args.config is None and not args.no_c3 and not args.batch and args.impl == "ours"
    if args.config is None:
        args.config = 2
    _claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
