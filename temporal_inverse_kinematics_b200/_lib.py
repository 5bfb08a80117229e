"""ctypes binding of libtik.so (include/tik.h).  No fallback: a missing library is an error."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TIK_LIB_PATH") or os.path.join(_HERE, "libtik.so")     # TIK_LIB_PATH: A/B builds of the same ABI (tools/)

HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "tik.h")


def _header_defines():
    """Integer #defines of include/tik.h: the header is the single source of the ABI's limits and codes."""
    import re
    out = {}
    with open(HEADER_PATH) as f:
        for m in re.finditer(r"^#define\s+(TIK_\w+)\s+\(?(-?\d+)\)?", f.read(), re.M):
            out[m.group(1)] = int(m.group(2))
    return out


_H = _header_defines()
TIK_F32, TIK_BF16 = _H["TIK_F32"], _H["TIK_BF16"]
MAX_BLOCKS, MAX_SLABS, MAX_JOINTS = _H["TIK_MAX_BLOCKS"], _H["TIK_MAX_SLABS"], _H["TIK_MAX_JOINTS"]
LBS_MAX_LANDMARKS = _H["TIK_LBS_MAX_LANDMARKS"]
ACT_NONE, ACT_RELU, ACT_LEAKY = 0, 1, 2
RES_NONE, RES_IDENTITY, RES_STEM, RES_CONV = 0, 1, 2, 3
OUT_NODE_MAJOR, OUT_TIME_MAJOR, OUT_ROWS_F32 = 0, 1, 2

vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float


class TikSlab(C.Structure):
    _fields_ = [("a_dev", vp), ("c", i32), ("t_in", i32), ("t_mul", i32), ("t_off", i32)]


class TikRowGemm(C.Structure):
    _fields_ = [("n_slabs", i32), ("slabs", TikSlab * MAX_SLABS), ("w_dev", vp), ("bias_dev", vp),
                ("bias_per_node", i32), ("nv", i64), ("v", i32), ("t_out", i32), ("c_out", i32),
                ("c_out_valid", i32), ("act", i32), ("slope", f32), ("res_kind", i32), ("res_dev", vp),
                ("res_w_dev", vp), ("res_cin", i32), ("res_t_mul", i32), ("res_t_in", i32), ("out_dev", vp),
                ("out_layout", i32)]


class TikWindowing(C.Structure):
    _fields_ = [("frames", i64), ("offset", i32), ("stride", i32), ("root_a", i32), ("root_b", i32)]


class TikBlock(C.Structure):
    _fields_ = [("c_in", i32), ("c_out", i32), ("stride", i32), ("kt", i32), ("res_kind", i32),
                ("agg_dev", vp), ("w_gcn_dev", vp), ("b_gcn_dev", vp), ("w_tcn_dev", vp), ("b_tcn_dev", vp),
                ("w_res_stem_dev", vp), ("res_as_slab", i32)]


class TikRawBN(C.Structure):
    _fields_ = [("weight_dev", vp), ("bias_dev", vp), ("mean_dev", vp), ("var_dev", vp), ("eps", C.c_double)]


class TikRawBlock(C.Structure):
    _fields_ = [("c_in", i32), ("c_out", i32), ("stride", i32), ("kt", i32), ("K", i32), ("V", i32), ("residual", i32),
                ("A_dev", vp), ("importance_dev", vp), ("gcn_w_dev", vp), ("gcn_b_dev", vp), ("bn1", TikRawBN),
                ("tcn_w_dev", vp), ("tcn_b_dev", vp), ("bn2", TikRawBN), ("res_w_dev", vp), ("res_b_dev", vp),
                ("bn_res", TikRawBN)]


class TikPackBuffers(C.Structure):
    _fields_ = [("agg_dev", vp), ("w_gcn_dev", vp), ("b_gcn_dev", vp), ("w_tcn_dev", vp), ("b_tcn_dev", vp),
                ("w_res_stem_dev", vp)]


class TikNet(C.Structure):
    _fields_ = [("V", i32), ("K", i32), ("c_in", i32), ("n_blocks", i32), ("in_scale_dev", vp),
                ("in_shift_dev", vp), ("blocks", TikBlock * MAX_BLOCKS), ("head_hidden", i32), ("head_out", i32),
                ("w1_dev", vp), ("b1_dev", vp), ("w2_dev", vp), ("b2_dev", vp), ("leaky_slope", f32)]


class TikLbsModel(C.Structure):
    _fields_ = [("V", i32), ("J", i32), ("kmax", i32), ("n_landmarks", i32), ("landmark_vid", i32 * LBS_MAX_LANDMARKS),
                ("v_shaped_dev", vp), ("rest_joints_dev", vp), ("posedirs_dev", vp), ("skin_idx_dev", vp), ("skin_w_dev", vp)]


_PROTOS = {
    "tik_version": (C.c_int, []),
    "tik_last_error": (C.c_char_p, []),
    "tik_check_device": (C.c_int, []),
    "tik_rot6d_to_rotmat": (C.c_int, [vp, vp, i64, vp]),
    "tik_aa_to_rotmat": (C.c_int, [vp, vp, i64, vp]),
    "tik_batch_rodrigues": (C.c_int, [vp, vp, i64, vp]),
    "tik_rotmat_to_aa": (C.c_int, [vp, vp, i64, C.c_int, vp]),
    "tik_quat_to_rotmat": (C.c_int, [vp, vp, i64, vp]),
    "tik_rotmat_to_quat": (C.c_int, [vp, vp, i64, vp]),
    "tik_quat_to_aa": (C.c_int, [vp, vp, i64, vp]),
    "tik_fk_body": (C.c_int, [vp, C.c_int, C.POINTER(f32), C.POINTER(i32), C.c_int, vp, vp, vp, vp, i64, vp]),
    "tik_lbs_workspace_bytes": (C.c_int, [C.POINTER(TikLbsModel), C.c_int, i64, C.POINTER(i64)]),
    "tik_lbs": (C.c_int, [C.POINTER(TikLbsModel), C.c_int, vp, vp, vp, C.c_int, vp, i64, vp, i64, vp, vp, C.c_int, vp]),
    "tik_stem_gcn": (C.c_int, [C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int, i64, C.c_int, C.c_int, C.c_int,
                               C.c_int, C.c_int, C.c_int, vp]),
    "tik_aggregate": (C.c_int, [C.c_int, vp, vp, vp, i64, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "tik_rowgemm": (C.c_int, [C.c_int, C.POINTER(TikRowGemm), vp]),
    "tik_gcn_fused": (C.c_int, [vp, vp, vp, vp, vp, i64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "tik_pack_bn": (C.c_int, [C.POINTER(TikRawBN), i64, vp, vp, vp]),
    "tik_pack_block_bytes": (C.c_int, [C.POINTER(TikRawBlock), C.c_int, C.c_int, C.POINTER(i64)]),
    "tik_pack_block": (C.c_int, [C.POINTER(TikRawBlock), C.c_int, C.c_int, C.POINTER(TikRawBN), C.POINTER(TikPackBuffers),
                                 C.POINTER(TikBlock), vp]),
    "tik_stgcn_out_frames": (C.c_int, [C.POINTER(TikNet), C.c_int]),
    "tik_stgcn_workspace_bytes": (C.c_int, [C.POINTER(TikNet), C.c_int, i64, i64, C.c_int, C.POINTER(i64)]),
    "tik_stgcn_plan_create": (C.c_int, [C.POINTER(TikNet), C.c_int, i64, i64, C.c_int, vp, i64, C.POINTER(vp)]),
    "tik_stgcn_plan_run": (C.c_int, [vp, vp, i64, vp, vp, vp]),
    "tik_stgcn_plan_run_windows": (C.c_int, [vp, vp, C.POINTER(TikWindowing), i64, vp, vp, vp]),
    "tik_stgcn_plan_profile": (C.c_int, [vp, vp, i64, vp, vp, C.POINTER(C.c_double), C.POINTER(i64), C.POINTER(C.c_double)]),
    "tik_stgcn_plan_launches": (i64, [vp, i64]),
    "tik_stgcn_plan_destroy": (None, [vp]),
    "tik_stgcn_latency_workspace_bytes": (C.c_int, [C.POINTER(TikNet), i64, C.c_int, C.POINTER(i64)]),
    "tik_stgcn_latency_create": (C.c_int, [C.POINTER(TikNet), i64, C.c_int, vp, i64, C.POINTER(vp)]),
    "tik_stgcn_latency_run": (C.c_int, [vp, vp, i64, vp, vp]),
    "tik_stgcn_latency_run_windows": (C.c_int, [vp, vp, C.POINTER(TikWindowing), i64, vp, vp]),
    "tik_stgcn_latency_phases": (C.c_int, [vp]),
    "tik_stgcn_latency_destroy": (None, [vp]),
    "tik_debug_latency_times": (C.c_int, [vp, vp]),
    "tik_debug_set_umma_shift": (C.c_int, [C.c_int, C.c_int]),
    "tik_debug_set_umma_times": (C.c_int, [vp]),
}

_lib = None


def exported_symbols():
    """Names declared in include/tik.h (used by the CPU-side ABI test)."""
    return sorted(_PROTOS)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m temporal_inverse_kinematics_b200.build` "
                "(there is no CPU or PyTorch fallback for the CUDA path)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().tik_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libtik error {rc}: {msg}")


def ptr(t):
    """Device (or host) address of a tensor, or None."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def on_device(t):
    """Context manager making the tensor's (or torch.device's) GPU the current CUDA device for the enclosed libtik
    calls: kernels, function attributes, cudaGetDevice and the plan's setup copies all act on the *current* device,
    which need not be the one the caller's tensors live on (a model on cuda:1 while cuda:0 is current)."""
    import torch
    dev = t.device if torch.is_tensor(t) else t
    if dev.index is None or dev.index == torch.cuda.current_device():
        return _NULL_CTX                       # already current: entering torch.cuda.device costs ~10 us per call
    return torch.cuda.device(dev)


class _NullCtx:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


_NULL_CTX = _NullCtx()
