"""ctypes binding of lib/libacr_b200.so (C ABI declared in /include/acr_b200.h).

There is deliberately no fallback: if the shared library is missing or a call fails, an
exception is raised.  Nothing here imports the oracle.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
# ACR_B200_LIB selects a variant build (tools/build_variant.py, A/B measurements); the product library is the default
LIB_PATH = os.environ.get("ACR_B200_LIB") or os.path.join(os.path.dirname(_HERE), "lib", "libacr_b200.so")

OK = 0
OP_STEM, OP_CONV, OP_FUSE, OP_BILINEAR2X, OP_COORD, OP_POOL, OP_PARTHEAD, OP_CONV_REF, OP_FINALCONV, OP_IM2COL_STEM, OP_STEM_TC = range(1, 12)
DT_BF16, DT_F16, DT_F32, DT_U8 = 0, 1, 2, 3


class AcrB200Error(RuntimeError):
    pass


class Map(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("pix_stride", C.c_int)]


class ParseOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "params_pred", "cam", "global_orient", "hand_pose", "betas", "poses", "detection_flag",
        "reorganize_idx", "batch_ids", "centers_pred", "centers_conf", "hand_type", "offsets_out",
        "counts", "top_idx", "top_score", "row_src")]


class Tensor(C.Structure):
    _fields_ = [("offset", C.c_uint64), ("C", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
                ("pix_stride", C.c_int32), ("dtype", C.c_int32), ("external", C.c_int32)]


class Op(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_in", C.c_int32), ("out", Tensor), ("in_", Tensor * 4),
                ("aux", Tensor * 4), ("w_offset", C.c_uint64 * 12),
                ("k", C.c_int32), ("stride", C.c_int32), ("relu", C.c_int32), ("has_residual", C.c_int32),
                ("cin_pad", C.c_int32), ("cout_pad", C.c_int32), ("shift", C.c_int32 * 4),
                ("stream_id", C.c_int32), ("wait_mask", C.c_int32), ("fparam", C.c_float * 4)]


class Gather(C.Structure):
    """acr_b200_gather (include/acr_b200.h): symmetric gather allocation of the fused vertex all-gather."""
    _fields_ = [("peer_base", C.c_uint64 * 8), ("multicast_base", C.c_uint64), ("world", C.c_int32), ("rank", C.c_int32),
                ("rows", C.c_int64), ("slot_bytes", C.c_uint64), ("counts_offset", C.c_uint64), ("flags_offset", C.c_uint64),
                ("local_state", C.c_void_p)]


_lib: Optional[C.CDLL] = None

EXPORTS = ["acr_b200_last_error", "acr_b200_version", "acr_b200_mano_model_floats", "acr_b200_mano_pack_model",
           "acr_b200_mano_forward", "acr_b200_mano_forward_gather", "acr_b200_gather_wait", "acr_b200_cam_trans", "acr_b200_preprocess", "acr_b200_one_euro_state_floats", "acr_b200_one_euro_smooth",
           "acr_b200_one_euro_smooth_streams", "acr_b200_rot6d_to_aa", "acr_b200_rodrigues", "acr_b200_parse",
           "acr_b200_parse_per_frame",
           "acr_b200_plan_create", "acr_b200_plan_run", "acr_b200_plan_profile", "acr_b200_plan_num_launches", "acr_b200_plan_destroy",
           "acr_b200_run_op", "acr_b200_conv_describe", "acr_b200_pack_conv"]

# acr_b200_conv_describe: field order of its info array (ACR_CONV_INFO_* in include/acr_b200.h)
CONV_INFO = ("ck", "mode", "b_resident", "nsplit", "nsub", "nbuf", "epilogue", "epi_nb", "SA", "SB", "grid", "vtiles")
MODE_PATCH, MODE_RESIDENT, MODE_XPAIR, MODE_DIAG, MODE_P1, MODE_S2X = 1, 2, 4, 8, 16, 32


def load() -> C.CDLL:
    """Load the shared library (once).  Fails loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AcrB200Error(f"{LIB_PATH} not found: build it with `python -m acr_b200.build` "
                           "(or __graft_entry__.build()); there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    vp, i32, f32 = C.c_void_p, C.c_int, C.c_float
    lib.acr_b200_last_error.restype = C.c_char_p
    lib.acr_b200_version.restype = C.c_char_p
    lib.acr_b200_mano_model_floats.restype = C.c_size_t
    lib.acr_b200_mano_pack_model.argtypes = [vp] * 6 + [i32, vp]
    lib.acr_b200_mano_forward.argtypes = [vp, vp, vp, vp, vp, i32, vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.acr_b200_mano_forward_gather.argtypes = [vp, vp, vp, vp, vp, i32, vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp,
                                                 vp, C.POINTER(Gather), vp]
    lib.acr_b200_gather_wait.argtypes = [C.POINTER(Gather), vp]
    lib.acr_b200_cam_trans.argtypes = [vp, vp, vp, i32, f32, f32, vp, vp]
    lib.acr_b200_preprocess.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, i32, i32, i32, i32, vp, vp]
    lib.acr_b200_one_euro_state_floats.restype = C.c_size_t
    lib.acr_b200_one_euro_smooth.argtypes = [vp, vp, vp, vp, vp, i32, vp, f32, vp]
    lib.acr_b200_one_euro_smooth_streams.argtypes = [vp, vp, vp, vp, vp, vp, i32, vp, i32, vp, f32, vp]
    lib.acr_b200_rot6d_to_aa.argtypes = [vp, i32, vp, vp]
    lib.acr_b200_rodrigues.argtypes = [vp, i32, vp, vp]
    lib.acr_b200_parse.argtypes = [Map] * 6 + [i32, f32, vp, vp, ParseOut, vp]
    lib.acr_b200_parse_per_frame.argtypes = [Map] * 6 + [i32, f32, vp, vp, ParseOut, vp]
    lib.acr_b200_plan_create.argtypes = [C.POINTER(Op), i32, i32, vp, C.c_size_t, vp, C.c_size_t, i32,
                                         C.POINTER(vp)]
    lib.acr_b200_plan_run.argtypes = [vp, vp, vp]
    lib.acr_b200_plan_profile.argtypes = [vp, vp, vp, vp, vp]
    lib.acr_b200_plan_num_launches.argtypes = [vp]
    lib.acr_b200_plan_destroy.argtypes = [vp]
    lib.acr_b200_plan_destroy.restype = None
    lib.acr_b200_run_op.argtypes = [C.POINTER(Op), i32, vp, vp, vp, i32, vp]
    lib.acr_b200_conv_describe.argtypes = [C.POINTER(Op), i32, vp, vp, i32, vp, i32]
    lib.acr_b200_pack_conv.argtypes = [vp] * 6 + [f32, i32, i32, i32, i32, i32, i32, vp, vp]
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != OK:
        msg = load().acr_b200_last_error().decode(errors="replace")
        raise AcrB200Error(f"{what or 'acr_b200 call'} failed (rc={rc}): {msg}")


def ptr(t) -> Optional[int]:
    """Raw device (or host) pointer of a torch tensor / numpy array, None passes through."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


def current_stream(device=None) -> int:
    """cudaStream_t of torch's current stream on `device` (default: the current device)."""
    import torch
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(*tensors):
    """All non-None arguments must be CUDA tensors on ONE device; returns that device (None if no tensor).
    The kernels are launched on that device's current stream, under a device guard (`on(dev)`), so ops on
    tensors of a non-current device do not end up on the wrong device / stream."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise AcrB200Error("acr_b200 kernels need CUDA tensors; there is no CPU fallback on the product path")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise AcrB200Error(f"acr_b200: arguments live on different devices ({dev} and {t.device})")
    return dev


def on(device):
    """Context manager: make `device` current for the launches inside (cudaFuncSetAttribute, events and the
    launch itself are per device)."""
    import torch
    return torch.cuda.device(device)
