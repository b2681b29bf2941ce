"""Pose smoothing of the demo's output path: lib/utils/smooth_pose.py with lib/utils/one_euro_filter.py, on the device.

The reference filters a person's 72 pose values with a One-Euro filter in numpy (frame 0 passes through, then one filter call
per frame with t_e = 1) and re-runs SMPL once per frame at batch 1.  Here the filter is one launch of tp_one_euro_filter
(csrc/smooth.cu; bit-identical to the reference's float32 arithmetic) and SMPL is one call over all frames.

    verts, pose_hat, joints3d = smooth_pose(pred_pose [N,72], pred_betas [N,10], min_cutoff=0.004, beta=0.7,
                                            smpl=model.regressor.smpl)

The same kernel runs per frame inside tepose_b200.tracks (TrackedTePose(..., smooth=(min_cutoff, beta))), with the filter
state of each slot kept on the device between pushes.
"""
from __future__ import annotations

import math

import torch

from . import _native as nv
from .smpl import SMPL, SMPL_MODEL_DIR, smpl_forward_native

POSE = 72                               # theta[:, 3:75]: global orientation + 23 body joints, axis-angle
SMOOTH_KEYS = ("pose_smooth", "verts_smooth", "joints3d_smooth")


def smooth_params(smooth):
    """smooth= of TrackedTePose: None, or (min_cutoff, beta), two finite non-negative numbers -> (float, float)."""
    if smooth is None:
        return None
    try:
        vals = tuple(smooth)
    except TypeError:
        raise ValueError(f"smooth must be None or (min_cutoff, beta), got {smooth!r}") from None
    if len(vals) != 2 or not all(isinstance(v, (int, float)) and not isinstance(v, bool) for v in vals):
        raise ValueError(f"smooth must be None or (min_cutoff, beta), two numbers, got {smooth!r}")
    if not all(math.isfinite(v) and v >= 0 for v in vals):
        raise ValueError(f"smooth (min_cutoff, beta) must be finite and >= 0, got {smooth!r}")
    return float(vals[0]), float(vals[1])


def one_euro_filter(x, out, state, count, reset, K, min_cutoff, beta):
    """One tp_one_euro_filter launch over S = state.shape[0] sequences of C = state.shape[2] channels.  x / out: sequence s, row r
    at s*stride(0) + r*stride(1) (column views allowed; for 2-D views the row stride is the sequence stride); state [S,2,C];
    count / reset int32 [S] on the device."""
    S, _, C = state.shape
    ld = lambda t: (t.stride(0), t.stride(1) if t.dim() == 3 else t.stride(0))
    (sx, rx), (so, ro) = ld(x), ld(out)
    for t in (x, out, state, count, reset):
        nv.require_cuda(t)
    nv.check(nv.lib().tp_one_euro_filter(nv.vp(x.data_ptr()), sx, rx, nv.vp(out.data_ptr()), so, ro, nv.ptr(state),
                                         nv.vp(count.data_ptr()), nv.vp(reset.data_ptr()), S, K, C, min_cutoff, beta,
                                         nv.stream()), "tp_one_euro_filter")


def smpl_rows(smpl: SMPL, pose, betas, n: int):
    """SMPL.forward(pose2rot=True) of n rows: pose [n,72] axis-angle and betas [n,10] (row strides as given, columns contiguous)
    -> vertices [n,6890,3], joints [n,49,3], through the same native call and joint tables as SMPL.forward."""
    p = smpl.packed()
    verts, joints, _, _, _ = smpl_forward_native(p, pose, pose.stride(0), nv.POSE_AXIS_ANGLE, betas, betas.stride(0), None, 0, n,
                                                 smpl._jreg_extra, smpl._src49, want_theta=False, want_rotmat=False,
                                                 blend_mode=1 if smpl.blend_precision == "bf16" else 0)
    return verts, joints


def _rows(t, dev):
    """t as fp32 rows with contiguous columns on dev: a view such as theta[:, 3:75] is passed as it is (the kernels take row
    strides), anything else is copied."""
    if t.device == torch.device(dev) and t.dtype == torch.float32 and t.stride(1) == 1 and t.stride(0) >= t.shape[1]:
        return t
    return t.to(dev, torch.float32).contiguous()


@torch.no_grad()
@nv.device_guard
def smooth_pose(pred_pose: torch.Tensor, pred_betas: torch.Tensor, min_cutoff=0.004, beta=0.7, smpl=None):
    """Drop-in for lib/utils/smooth_pose.py:smooth_pose on CUDA tensors: pred_pose [N,72] (theta[:, 3:75]) and pred_betas [N,10]
    -> (verts [N,6890,3], pose_hat [N,72], joints3d [N,49,3]).  Row 0 passes through; every later row is the reference's
    One-Euro filter at t_e = 1.  smpl: the SMPL module to use (normally model.regressor.smpl); None builds SMPL(SMPL_MODEL_DIR)
    on the device of pred_pose, as the reference builds its own."""
    nv.require_cuda(pred_pose, "pred_pose")
    if pred_pose.dim() != 2 or pred_pose.shape[1] != POSE or pred_pose.shape[0] < 1:
        raise ValueError(f"expected pred_pose [N>=1,{POSE}], got {tuple(pred_pose.shape)}")
    N = pred_pose.shape[0]
    if tuple(pred_betas.shape) != (N, 10):
        raise ValueError(f"expected pred_betas [{N},10], got {tuple(pred_betas.shape)}")
    min_cutoff, beta = smooth_params((min_cutoff, beta))
    dev = pred_pose.device
    if smpl is None:
        smpl = SMPL(SMPL_MODEL_DIR, batch_size=1, create_transl=False).to(dev)
    x, betas = _rows(pred_pose, dev), _rows(pred_betas, dev)
    pose_hat = torch.empty(N, POSE, device=dev)
    state = torch.empty(1, 2, POSE, device=dev)
    table = torch.tensor([N, 1], dtype=torch.int32).to(dev)                       # count | reset of the one sequence
    one_euro_filter(x, pose_hat, state, table[0:1], table[1:2], N, min_cutoff, beta)
    verts, joints = smpl_rows(smpl, pose_hat, betas, N)
    return verts, pose_hat, joints
