"""Sequence-level inference with the reference's call signature (reference inference.py:37-67), entirely on the GPU.

The reference builds one edge-padded, root-centred window per frame on the host (InferenceDataset, numpy per item),
collates them with a DataLoader (batch 64), runs the model batch by batch with a D2H copy each, and averages the
window predictions per frame in Python lists.  Here the sequence is uploaded once, the windows are *never
materialised* (the stem kernel gathers frames with clamped indices and subtracts the mid-hip root on the fly), all
windows go through the network in one pass, and the per-frame aggregation runs on the device.

`run_inference_batch` does the same for a list of sequences at once: they are packed into one buffer, the windows of
every sequence go through one pass (each window clamped to its own sequence's frames), and one kernel takes the
per-frame means of all of them.
"""
import numpy as np
import torch

from .keypoints_util import COCO_ROOT_PAIR


def _window_sum(vals, h_w_size):
    """sum and count over the windows that cover each frame: window i contributes vals[i, o + h] to frame i + o."""
    F = vals.shape[0]
    acc = torch.zeros((F,) + tuple(vals.shape[2:]), dtype=vals.dtype, device=vals.device)
    cnt = torch.zeros((F,) + (1,) * (vals.dim() - 2), dtype=vals.dtype, device=vals.device)
    for o in range(-h_w_size, h_w_size + 1):
        lo, hi = max(o, 0), F + min(o, 0)                 # destination frames i + o
        if hi <= lo:
            continue
        acc[lo:hi] += vals[lo - o:hi - o, o + h_w_size]
        cnt[lo:hi] += 1
    return acc, cnt


def sequence_tables(lengths, win_frames, offset, stride):
    """Tables of a ragged batch of sequences packed back to back (include/tik.h TikSeqBatch): int64 numpy arrays
    frame_start and window_start of len(lengths)+1 entries.  Sequence s has the windows forward_windows gives one
    sequence of F_s frames: F_s if offset < 0, else max(0, (F_s - win_frames - offset) // stride + 1)."""
    F = np.asarray([int(n) for n in lengths], dtype=np.int64)
    if F.size == 0:
        raise ValueError("lengths must name at least one sequence")
    if (F < 1).any():
        k = int(np.argmax(F < 1))
        raise ValueError(f"sequence {k} has length {int(F[k])}: every sequence needs at least one frame")
    if int(stride) < 1 or int(win_frames) < 1:
        raise ValueError("sequence_tables needs stride >= 1 and win_frames >= 1")
    W = F if offset < 0 else np.maximum(0, (F - int(win_frames) - int(offset)) // int(stride) + 1)
    zero = np.zeros(1, dtype=np.int64)
    return np.concatenate([zero, np.cumsum(F)]), np.concatenate([zero, np.cumsum(W)]).astype(np.int64)


def packed_window_mean(preds, frame_start, h_w_size=0, mode="euclidean"):
    """window_mean of every sequence of a ragged batch in one kernel (`tik_window_mean`), with the frame_start table
    already on the device (int64, n_seqs+1 entries): the launch is all this does, so it can be captured in a CUDA
    graph.  preds (frames, T', D) CUDA fp32, one window per packed frame.  Arguments are checked by window_mean."""
    from . import _lib as L
    preds = preds.detach().float().contiguous()
    frames, Tp, D = preds.shape
    out = torch.empty((frames, D), dtype=torch.float32, device=preds.device)
    code = L.MEAN_ROTATION if mode == "rotation" else L.MEAN_EUCLIDEAN
    with L.on_device(preds):
        L.check(L.lib().tik_window_mean(L.ptr(preds), frames, Tp, D, L.ptr(frame_start), frame_start.numel() - 1,
                                        int(h_w_size), code, L.ptr(out), L.stream_ptr(preds.device)))
    return out


def window_mean(preds, h_w_size=0, mode="euclidean", lengths=None):
    """Per-frame mean of overlapping window predictions (reference inference.py:56-67).
    preds (F, T', D): window i contributes preds[i, o + h_w_size] to frame i + o for o in [-h_w_size, h_w_size].

    mode="euclidean" is the reference's ``np.mean`` of the axis-angle vectors.  mode="rotation" (SURVEY.md 8f row 2)
    averages ROTATIONS instead: every prediction goes axis-angle -> rotation matrix (`batch_rodrigues` kernel), the
    matrices are averaged per frame and joint, the mean is projected back onto SO(3) by Gram-Schmidt of its first two
    columns (the 6-D representation's mean; `rot6d_to_rotmat` kernel) and returned as axis-angle
    (`rotation_matrix_to_angle_axis` kernel).  Axis-angle vectors near +-pi of the same rotation average to ~0 in
    euclidean mode and to the right rotation here.

    lengths (host ints): preds holds the windows of several sequences packed back to back, one window per frame,
    sum(lengths) rows; each sequence is averaged on its own (a window never contributes to a neighbouring sequence)
    in one `tik_window_mean` launch.  The result equals torch.cat of window_mean per sequence: bit for bit in euclidean
    mode, to rounding in rotation mode."""
    if mode not in ("euclidean", "rotation"):
        raise ValueError("mode must be 'euclidean' or 'rotation'")
    if lengths is not None:
        if preds.dim() != 3:
            raise ValueError(f"expected (frames, T', D) predictions, got {tuple(preds.shape)}")
        frame_start, _ = sequence_tables(lengths, 1, -1, 1)
        if int(frame_start[-1]) != preds.shape[0]:
            raise ValueError(f"lengths sum to {int(frame_start[-1])} frames, preds has {preds.shape[0]} rows")
        if h_w_size < 0 or preds.shape[1] < 2 * h_w_size + 1:
            raise ValueError(f"need {2 * h_w_size + 1} predictions per window, the model emits {preds.shape[1]}")
        if mode == "rotation" and preds.shape[2] % 3:
            raise ValueError("rotation mode needs axis-angle predictions (D divisible by 3)")
        return packed_window_mean(preds, torch.from_numpy(frame_start).to(preds.device), h_w_size, mode)
    if h_w_size == 0:
        return preds[:, 0]
    if preds.shape[1] < 2 * h_w_size + 1:
        raise ValueError(f"need {2 * h_w_size + 1} predictions per window, the model emits {preds.shape[1]}")
    if mode == "euclidean":
        acc, cnt = _window_sum(preds, h_w_size)
        return acc / cnt
    from . import geometry
    F, Tp, D = preds.shape
    if D % 3:
        raise ValueError("rotation mode needs axis-angle predictions (D divisible by 3)")
    R = geometry.batch_rodrigues(preds.reshape(-1, 3)).view(F, Tp, D // 3, 9)
    acc, cnt = _window_sum(R, h_w_size)
    M = (acc / cnt).view(-1, 3, 3)
    x6 = M[:, :, :2].reshape(-1, 6)                        # (a1, a2) interleaved as rot6d_to_rotmat reads them
    return geometry.rotation_matrix_to_angle_axis(geometry.rot6d_to_rotmat(x6)).view(F, D)


def run_inference(model, seq_3d_kps, h_w_size=0, relative_pose=True, mean_mode="euclidean"):
    """model: IKPoseTrainer (or anything with .hparams.win_size, .regressor, .device); seq_3d_kps (F, 17, 3).
    Returns (F, 66) axis-angle poses as numpy, like the reference (`h_w_size` / `mean_mode`: see window_mean)."""
    seq = torch.as_tensor(np.asarray(seq_3d_kps, dtype=np.float32)).to(model.device).contiguous()
    half = model.hparams.win_size // 2
    poses = model.regressor.forward_windows(seq, 2 * half + 1, offset=-half, stride=1,
                                            root=COCO_ROOT_PAIR if relative_pose else None)["poses"]
    return window_mean(poses, h_w_size, mean_mode).detach().cpu().numpy()


def run_inference_batch(model, seqs, h_w_size=0, relative_pose=True, mean_mode="euclidean"):
    """run_inference over a list of sequences in one pass: returns the list of (F_s, 66) numpy arrays
    ``[run_inference(model, s, h_w_size, relative_pose, mean_mode) for s in seqs]`` (bit for bit in euclidean mode).
    The sequences go to the device in one copy, all their windows through one forward_windows(lengths=...), the
    per-frame means through one kernel, and the poses come back in one copy.  A loop of run_inference pays a
    nearly empty network pass and a host synchronisation per sequence; this pays them once."""
    arrs = [np.asarray(s, dtype=np.float32) for s in seqs]
    if not arrs:
        return []
    for k, a in enumerate(arrs):
        if a.ndim != 3 or a.shape[0] == 0:
            raise ValueError(f"sequence {k} has shape {a.shape}: every sequence needs at least one (V, C) frame")
    lengths = [a.shape[0] for a in arrs]
    packed = torch.from_numpy(np.concatenate(arrs)).to(model.device)
    half = model.hparams.win_size // 2
    poses = model.regressor.forward_windows(packed, 2 * half + 1, offset=-half, stride=1,
                                            root=COCO_ROOT_PAIR if relative_pose else None, lengths=lengths)["poses"]
    out = window_mean(poses, h_w_size, mean_mode, lengths=lengths).detach().cpu().numpy()
    return np.split(out, np.cumsum(lengths)[:-1])
