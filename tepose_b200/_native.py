"""ctypes binding of the C-ABI library declared in include/tepose_b200.h.

There is deliberately NO fallback: if libtepose_b200.so is missing, or a call is made
without a CUDA device, this raises -- the product never routes through torch ops or the
CPU oracle for the hot path.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# TEPOSE_B200_LIB selects another build of the same sources (tests: the -DTP_BARRIER_ACQUIRE_FENCE twin, tepose_b200/build.py)
LIB_PATH = os.environ.get("TEPOSE_B200_LIB") or os.path.join(_HERE, "libtepose_b200.so")

PRECISION_FP32, PRECISION_BF16, PRECISION_BF16X3 = 0, 1, 2
POSE_ROTMAT, POSE_AXIS_ANGLE, POSE_ROT6D = 0, 1, 2
RODRIGUES_SMPLX, RODRIGUES_QUAT = 0, 1
GEMM_RELU, GEMM_OUT_BF16, GEMM_OUT_SPLIT3, GEMM_RES_SPLIT3 = 1, 2, 4, 8      # tp_gemm_seg.flags
# "fp32_tc": fp32-grade results with the two big contractions (K1 input projection, K2 recurrence) on tensor cores as 3-term bf16
# splits (TP_PRECISION_BF16X3); every other stage runs exactly as in "fp32", which is the code the C ABI sees for them
PRECISIONS = {"fp32": PRECISION_FP32, "bf16": PRECISION_BF16, "fp32_tc": PRECISION_FP32}

# every symbol include/tepose_b200.h declares (tests check the library exports all of them)
EXPORTS = [
    "tp_version", "tp_last_error", "tp_launch_count", "tp_set_pdl", "tp_set_ief_cluster", "tp_device_info",
    "tp_rot6d_to_rotmat", "tp_rotmat_to_angle_axis", "tp_batch_rodrigues", "tp_projection",
    "tp_pack_rows", "tp_pack_rows_ex", "tp_pack_rows_f16", "tp_split3_bf16", "tp_unpack_rows_residual", "tp_gemm_f32", "tp_gemm_f32_splitk_workspace_bytes", "tp_gemm_f32_splitk",
    "tp_pack_mma_a_bytes", "tp_pack_mma_a_bf16", "tp_skinny_bf16_workspace_bytes", "tp_skinny_bf16", "tp_skinny_bf16_ex", "tp_gemm_bf16_tc",
    "tp_pack_whh_bf16", "tp_whh_umma_bytes", "tp_pack_whh_umma", "tp_gru_set_trace", "tp_gru_workspace_bytes", "tp_gru_recurrence", "tp_gru_recurrence_ex",
    "tp_encoder_heads_workspace_bytes", "tp_encoder_heads", "tp_encoder_heads_cat", "tp_ief_workspace_bytes", "tp_ief_forward", "tp_heads_ief_forward",
    "tp_smpl_workspace_bytes", "tp_smpl_forward", "tp_smpl_forward_ex",
    "tp_pose_metrics", "tp_accel_error", "tp_vertex_error",
    "tp_transpose_f32", "tp_colsum_f32", "tp_mask_scale", "tp_relu_backward", "tp_axpby_f32", "tp_gru_cell_backward",
    "tp_rot6d_backward", "tp_rotmat_to_angle_axis_backward", "tp_smpl_backward_workspace_bytes", "tp_smpl_backward",
    "tp_tepose_loss_workspace_bytes", "tp_tepose_loss",
    "tp_nchw_to_nhwc_bf16", "tp_im2col_nhwc_bf16", "tp_maxpool3x3s2_nhwc_bf16", "tp_avgpool_nhwc_bf16",
    "tp_crop_normalize_bf16",
    "tp_nchw_to_nhwc_split3", "tp_maxpool3x3s2_nhwc_split3", "tp_avgpool_nhwc_split3", "tp_crop_normalize_split3",
    "tp_window_slots_push", "tp_window_slots_commit",
    "tp_render_workspace_bytes", "tp_render_meshes",
    "tp_one_euro_filter",
]

vp, i32, i64, f32, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_size_t


class GemmSeg(C.Structure):
    _fields_ = [("m_start", i32), ("m_rows", i32), ("n_start", i32), ("n_cols", i32),
                ("out", vp), ("ldc", i64), ("bias", vp), ("flags", i32), ("ldr", i32), ("residual", vp)]


class Crop(C.Structure):
    _fields_ = [("frame", i32), ("cx", f32), ("cy", f32), ("w", f32), ("h", f32), ("scale", f32)]


class GruJob(C.Structure):
    _fields_ = [("gi", vp), ("ldg", i64), ("w_hh", vp), ("b_hh", vp), ("h0", vp),
                ("y", vp), ("ldy", i64), ("y_lp", vp), ("ldy_lp", i64),
                ("h_final", vp), ("ld_hf", i64), ("steps", i32),
                ("t_in0", i32), ("t_in_step", i32), ("t_out0", i32), ("t_out_step", i32), ("gates", vp), ("w_hh_umma", vp)]


class IefWeights(C.Structure):
    _fields_ = [(n, vp) for n in ("w1x", "b1", "w1p", "w2", "b2", "wdec", "bdec")]


class SmplModel(C.Structure):
    _fields_ = [("blend", vp), ("j_template", vp), ("j_shapedirs", vp), ("parents", vp),
                ("skin_idx", vp), ("skin_w", vp), ("ks", i32), ("n_verts", i32), ("vp", i32),
                ("blend_tc", vp), ("template_pad", vp), ("blend_km", vp), ("blend_um", vp), ("skin_um", vp)]


class SmplRegFold(C.Structure):
    _fields_ = [("m_km", vp), ("q_bias", vp), ("g0", vp), ("nreg", i32), ("nq_pad", i32)]


_SIGNATURES = {
    "tp_version": (C.c_int, []),
    "tp_last_error": (C.c_char_p, []),
    "tp_launch_count": (C.c_ulonglong, []),
    "tp_set_pdl": (C.c_int, [C.c_int]),
    "tp_set_ief_cluster": (C.c_int, [C.c_int]),
    "tp_nchw_to_nhwc_bf16": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "tp_im2col_nhwc_bf16": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "tp_maxpool3x3s2_nhwc_bf16": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "tp_avgpool_nhwc_bf16": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, vp]),
    "tp_crop_normalize_bf16": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, vp]),
    "tp_nchw_to_nhwc_split3": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "tp_maxpool3x3s2_nhwc_split3": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "tp_avgpool_nhwc_split3": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, vp]),
    "tp_crop_normalize_split3": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, vp]),
    "tp_window_slots_push": (C.c_int, [vp, C.c_int, C.c_int, i64, vp, vp, vp, vp]),
    "tp_window_slots_commit": (C.c_int, [vp, C.c_int, C.c_int, i64, vp, vp, vp]),
    "tp_one_euro_filter": (C.c_int, [vp, i64, i64, vp, i64, i64, vp, vp, vp, C.c_int, C.c_int, C.c_int, f32, f32, vp]),
    "tp_render_workspace_bytes": (sz, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "tp_render_meshes": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, sz, vp]),
    "tp_device_info": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(sz)]),
    "tp_rot6d_to_rotmat": (C.c_int, [vp, vp, i64, vp]),
    "tp_rotmat_to_angle_axis": (C.c_int, [vp, vp, i64, vp]),
    "tp_batch_rodrigues": (C.c_int, [vp, vp, i64, C.c_int, vp]),
    "tp_projection": (C.c_int, [vp, vp, vp, C.c_int, C.c_int, vp]),
    "tp_pack_rows_f16": (C.c_int, [vp, i64, i64, C.c_int, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_int, vp, sz, vp]),
    "tp_split3_bf16": (C.c_int, [vp, i64, C.c_int, C.c_int, vp, vp]),
    "tp_pack_rows": (C.c_int, [vp, i64, i64, C.c_int, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_int, vp]),
    "tp_pack_rows_ex": (C.c_int, [vp, i64, i64, C.c_int, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_int, vp, sz, vp]),
    "tp_heads_ief_forward": (C.c_int, [vp, vp, vp, i64, C.c_int, C.POINTER(IefWeights), C.c_int, vp, C.c_int, C.c_int, vp, vp, sz, vp, vp]),
    "tp_pose_metrics": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp]),
    "tp_accel_error": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]),
    "tp_vertex_error": (C.c_int, [vp, vp, C.c_int, C.c_int, vp, vp]),
    "tp_unpack_rows_residual": (C.c_int, [vp, i64, vp, i64, i64, C.c_int, C.c_int, C.c_int, vp, vp, vp]),
    "tp_gemm_f32": (C.c_int, [vp, i64, vp, i64, vp, vp, i64, vp, i64, C.c_int, C.c_int, C.c_int, f32, f32, C.c_int, vp]),
    "tp_gemm_f32_splitk_workspace_bytes": (sz, [C.c_int, C.c_int, C.c_int]),
    "tp_gemm_f32_splitk": (C.c_int, [vp, i64, vp, i64, vp, vp, i64, vp, i64, C.c_int, C.c_int, C.c_int, f32, f32, C.c_int,
                                     C.c_int, vp, sz, vp]),
    "tp_pack_mma_a_bytes": (sz, [C.c_int, C.c_int]),
    "tp_pack_mma_a_bf16": (C.c_int, [vp, i64, C.c_int, C.c_int, vp, vp]),
    "tp_skinny_bf16_workspace_bytes": (sz, [C.c_int, C.c_int, C.c_int]),
    "tp_skinny_bf16": (C.c_int, [vp, i64, C.c_int, C.c_int, vp, C.c_int, vp, vp, i64, vp, i64, f32, f32, C.c_int, C.c_int,
                                 vp, sz, vp]),
    "tp_skinny_bf16_ex": (C.c_int, [vp, i64, vp, i64, C.c_int, C.c_int, vp, C.c_int, vp, vp, i64, vp, i64, vp, i64, f32, f32,
                                    C.c_int, C.c_int, C.c_int, vp, sz, vp]),
    "tp_gemm_bf16_tc": (C.c_int, [vp, C.c_int, vp, C.c_int, C.c_int, C.POINTER(GemmSeg), C.c_int, vp]),
    "tp_pack_whh_bf16": (C.c_int, [vp, vp, C.c_int, vp]),
    "tp_whh_umma_bytes": (sz, [C.c_int]),
    "tp_pack_whh_umma": (C.c_int, [vp, vp, C.c_int, vp]),
    "tp_gru_set_trace": (None, [vp]),
    "tp_gru_workspace_bytes": (sz, [C.c_int, C.c_int, C.c_int]),
    "tp_gru_recurrence": (C.c_int, [C.POINTER(GruJob), C.c_int, C.c_int, C.c_int, C.c_int, vp, sz, vp]),
    "tp_gru_recurrence_ex": (C.c_int, [C.POINTER(GruJob), C.c_int, C.c_int, C.c_int, C.c_int, vp, sz, vp, vp]),
    "tp_encoder_heads_workspace_bytes": (sz, [C.c_int]),
    "tp_encoder_heads": (C.c_int, [C.c_int, vp, vp, vp, vp, vp, i64, vp, i64, C.c_int, C.c_int, C.c_int, vp, vp, vp, sz, vp]),
    "tp_encoder_heads_cat": (C.c_int, [C.c_int, vp, vp, vp, i64, C.c_int, C.c_int, vp, vp, vp, sz, vp]),
    "tp_ief_workspace_bytes": (sz, [C.c_int]),
    "tp_ief_forward": (C.c_int, [C.c_int, C.POINTER(IefWeights), vp, vp, C.c_int, vp, C.c_int, C.c_int, vp, vp, sz, vp]),
    "tp_transpose_f32": (C.c_int, [vp, i64, C.c_int, C.c_int, vp, i64, C.c_int, C.c_int, C.c_int, vp]),
    "tp_colsum_f32": (C.c_int, [vp, i64, C.c_int, C.c_int, vp, f32, vp]),
    "tp_mask_scale": (C.c_int, [vp, i64, vp, i64, C.c_int, C.c_int, f32, vp]),
    "tp_relu_backward": (C.c_int, [vp, i64, vp, i64, C.c_int, C.c_int, vp]),
    "tp_axpby_f32": (C.c_int, [vp, i64, vp, i64, C.c_int, C.c_int, f32, f32, vp]),
    "tp_gru_cell_backward": (C.c_int, [vp, i64, vp, i64, vp, i64, vp, i64, vp, i64, C.c_int, C.c_int, vp]),
    "tp_rot6d_backward": (C.c_int, [vp, vp, vp, i64, vp]),
    "tp_rotmat_to_angle_axis_backward": (C.c_int, [vp, vp, i64, C.c_int, vp, i64, C.c_int, vp]),
    "tp_smpl_backward_workspace_bytes": (sz, [C.POINTER(SmplModel), C.c_int]),
    "tp_smpl_backward": (C.c_int, [C.POINTER(SmplModel), C.c_int, vp, vp, i64, vp, i64, vp, C.c_int, vp, C.c_int, vp,
                                   vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
    "tp_tepose_loss_workspace_bytes": (sz, [C.c_int, C.c_int, C.c_int]),
    "tp_tepose_loss": (C.c_int, [vp, vp, C.c_int, vp, vp, C.c_int, vp, vp, C.c_int, C.POINTER(f32), vp, vp, vp, vp, vp, sz, vp]),
    "tp_smpl_workspace_bytes": (sz, [C.POINTER(SmplModel), C.c_int, C.c_int, C.c_int]),
    "tp_smpl_forward_ex": (C.c_int, [C.POINTER(SmplModel), C.c_int, vp, i64, C.c_int, vp, i64, vp, i64,
                                     vp, C.c_int, C.POINTER(SmplRegFold), vp, C.c_int, vp, vp, vp, vp, vp, C.c_int, vp, sz, vp]),
    "tp_smpl_forward": (C.c_int, [C.POINTER(SmplModel), C.c_int, vp, i64, C.c_int, vp, i64, vp, i64,
                                  vp, C.c_int, vp, C.c_int, vp, vp, vp, vp, vp, C.c_int, vp, sz, vp]),
}

_lib = None


def lib() -> C.CDLL:
    """Loads the native library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m tepose_b200.build` "
                "(or __graft_entry__.build()).  tepose_b200 has no CPU / torch fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().tp_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"tepose_b200 native call {what} failed (code {rc}): {msg}")


def require_cuda(t: torch.Tensor, name: str = "tensor") -> None:
    if not t.is_cuda:
        raise RuntimeError(f"tepose_b200: {name} must live on a CUDA device (got {t.device}); "
                           "there is no CPU path")


def ptr(t, dtype=None) -> vp:
    """Device pointer of a contiguous CUDA tensor (or NULL for None)."""
    if t is None:
        return vp(0)
    require_cuda(t)
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"expected {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError("tensor must be contiguous")
    return vp(t.data_ptr())


def stream() -> vp:
    return vp(torch.cuda.current_stream().cuda_stream)


def device_guard(fn):
    """Decorator for the public entry points: makes the device of the first CUDA tensor argument (else of the module's own
    parameters / buffers) the CURRENT device for the duration of the call.  The C ABI takes raw pointers and a stream; the stream
    (`stream()`), the workspaces, the SM count and the occupancy queries behind the cooperative launches all refer to the current
    device, so a model on cuda:1 called while cuda:0 is current would otherwise launch on the wrong device (ATen guards this for
    torch modules; the reference's modules therefore work in that situation, and so must their drop-ins)."""
    import functools

    @functools.wraps(fn)
    def wrapped(*args, **kwargs):
        dev = None
        for a in list(args) + list(kwargs.values()):
            if torch.is_tensor(a) and a.is_cuda:
                dev = a.device
                break
        if dev is None and args and isinstance(args[0], torch.nn.Module):
            t = next(iter(args[0].parameters()), None)
            if t is None:
                t = next(iter(args[0].buffers()), None)
            if t is not None and t.is_cuda:
                dev = t.device
        if dev is None or dev.index is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapped


def workspace(nbytes: int, device) -> torch.Tensor:
    """256-byte aligned scratch (torch's caching allocator aligns to 512 B)."""
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


# ---- optional stage markers (bench.py's per-kernel timing): CUDA events on the current stream
_marks = None


def start_marks():
    global _marks
    _marks = []


def stop_marks():
    global _marks
    out, _marks = _marks, None
    return out


def mark(name: str) -> None:
    if _marks is not None:
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        _marks.append((name, ev))


def pack_linear(w: torch.Tensor, precision: str) -> torch.Tensor:
    """nn.Linear weight [N,K] -> the operand layout the K3 kernels stream for `precision`:
    fp32: contiguous fp32 as is; bf16: tensor-core fragment order (tp_pack_mma_a_bf16)."""
    w = w.detach().float().contiguous()
    if precision != "bf16":
        return w
    n, k = w.shape
    out = torch.empty(lib().tp_pack_mma_a_bytes(n, k), dtype=torch.uint8, device=w.device)
    check(lib().tp_pack_mma_a_bf16(ptr(w), k, n, k, ptr(out), stream()), "tp_pack_mma_a_bf16")
    return out
