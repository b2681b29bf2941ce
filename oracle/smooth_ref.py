"""Restatement of the reference's pose smoothing: lib/utils/one_euro_filter.py and lib/utils/smooth_pose.py (as TePose carries
them from VIBE), in numpy float32 as the reference computes them, with SMPL through oracle.torch_ref.smpl_forward.

one_euro_f32 is the same filter written out per channel with every float32 operation rounded on its own; it is the arithmetic
tp_one_euro_filter (tepose_b200/csrc/smooth.cu) implements, and tests/test_smooth.py holds it bit-identical to the class.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import torch_ref


# ---------------------------------------------------------------------------------------------------- lib/utils/one_euro_filter.py
def smoothing_factor(t_e, cutoff):
    r = 2 * math.pi * cutoff * t_e
    return r / (r + 1)


def exponential_smoothing(a, x, x_prev):
    return a * x + (1 - a) * x_prev


class OneEuroFilter:
    def __init__(self, t0, x0, dx0=0.0, min_cutoff=1.0, beta=0.0, d_cutoff=1.0):
        self.min_cutoff = float(min_cutoff)
        self.beta = float(beta)
        self.d_cutoff = float(d_cutoff)
        self.x_prev = x0
        self.dx_prev = float(dx0)
        self.t_prev = t0

    def __call__(self, t, x):
        t_e = t - self.t_prev
        a_d = smoothing_factor(t_e, self.d_cutoff)
        dx = (x - self.x_prev) / t_e
        dx_hat = exponential_smoothing(a_d, dx, self.dx_prev)
        cutoff = self.min_cutoff + self.beta * np.abs(dx_hat)
        a = smoothing_factor(t_e, cutoff)
        x_hat = exponential_smoothing(a, x, self.x_prev)
        self.x_prev = x_hat
        self.dx_prev = dx_hat
        self.t_prev = t
        return x_hat


# ---------------------------------------------------------------------------------------------------- lib/utils/smooth_pose.py
def filter_pose(pred_pose, min_cutoff=0.004, beta=0.7):
    """The filter part of smooth_pose: pred_pose [N,72] float32 -> pose_hat [N,72] float32 (row 0 unchanged, then one filter
    call per row at t = row index)."""
    pred_pose = np.asarray(pred_pose, np.float32)
    f = OneEuroFilter(np.zeros_like(pred_pose[0]), pred_pose[0], min_cutoff=min_cutoff, beta=beta)
    pose_hat = np.zeros_like(pred_pose)
    pose_hat[0] = pred_pose[0]
    for idx, pose in enumerate(pred_pose[1:]):
        idx += 1
        t = np.ones_like(pose) * idx
        pose_hat[idx] = f(t, pose)
    return pose_hat


def smooth_pose(m: "torch_ref.SmplModel", pred_pose, pred_betas, min_cutoff=0.004, beta=0.7):
    """smooth_pose(pred_pose [N,72], pred_betas [N,10]) with the SMPL model m: the filter, then SMPL once per frame at batch 1
    (the reference splits the orientation at index 1, which smplx undoes by concatenating before Rodrigues, so the row goes in
    as one 72-value axis-angle pose).  Returns (verts [N,V,3], pose_hat [N,72], joints3d [N,49,3]) as numpy float32."""
    pose_hat = filter_pose(pred_pose, min_cutoff, beta)
    betas = np.asarray(pred_betas, np.float32)
    verts, joints = [], []
    for idx in range(pose_hat.shape[0]):
        v, j, _ = torch_ref.smpl_forward(m, torch.from_numpy(betas[idx:idx + 1]), pose_aa=torch.from_numpy(pose_hat[idx:idx + 1]))
        verts.append(v.numpy())
        joints.append(j.numpy())
    return np.vstack(verts), pose_hat, np.vstack(joints)


# ---------------------------------------------------------------------------------------------------- the kernel's arithmetic
K_2PI = np.float32(2 * math.pi)


def one_euro_f32(x, min_cutoff, beta, state=None):
    """x [n,C] float32 filtered at t_e = 1 with every operation rounded on its own.  state None: row 0 passes through and starts
    the state; else (x_prev [C], dx_prev [C]) to continue from.  Returns (out [n,C], (x_prev, dx_prev))."""
    f32 = np.float32
    x = np.asarray(x, f32)
    out = np.empty_like(x)
    a_d = K_2PI / (K_2PI + f32(1))
    mc, b = f32(min_cutoff), f32(beta)
    t0 = 0
    if state is None:
        x_prev, dx_prev = x[0].copy(), np.zeros(x.shape[1], f32)
        out[0] = x[0]
        t0 = 1
    else:
        x_prev, dx_prev = (np.asarray(v, f32).copy() for v in state)
    for t in range(t0, x.shape[0]):
        dx = x[t] - x_prev
        dx_hat = a_d * dx + (f32(1) - a_d) * dx_prev
        cutoff = mc + b * np.abs(dx_hat)
        r = K_2PI * cutoff
        a = r / (r + f32(1))
        x_hat = a * x[t] + (f32(1) - a) * x_prev
        out[t], x_prev, dx_prev = x_hat, x_hat, dx_hat
    return out, (x_prev, dx_prev)
