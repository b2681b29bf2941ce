"""Frames to meshes on the device: the reference demo's per-frame loop (demo.py:183-252) from RGB frames and tracker boxes.

The reference crops every box on the host with cv2 (lib/data_utils/_img_utils.py: get_single_image_crop_demo), runs HMR's
feature extractor on the crops, bootstraps with VIBE and then runs TePose on a sliding T-frame window.  Here a frame's B crops
are cut and normalised by one kernel (tp_crop_normalize_bf16, bit-identical to the cv2 / torchvision crop rounded to bf16), the
features go straight into the window's feature ring, and once the window is full every frame is ONE CUDA-graph replay:

    crop -> HMR ResNet-50 (76 launches) -> feature roll -> TePose window step -> theta roll

The window, both rings and the step body are tepose_b200.stream.WindowedTePose's.  The crop table is device memory read by the
graph, so boxes may change on every frame.

    vt = VideoTePose(hmr, model, model_vibe, J_regressor=J, batch=B)      # B tracked people (or B cameras)
    for frames, crops in video:                   # frames uint8 [F,H,W,3] RGB, crops [B,6] rows (frame, cx, cy, w, h, scale)
        out = vt.push(frames, crops)              # None, None, ..., then frames 0..T-1, then one frame per push
  or a whole clip:
    out = vt.run(frames [N,H,W,3], crops [B,N,6])  # {theta [B,N,85], verts [B,N,6890,3], ...}
"""
from __future__ import annotations

import torch

from . import _native as nv
from .hmr import CROP, CROP_FIELDS, make_crop_table
from .stream import FEAT, OUTPUT_KEYS, WindowedTePose


class VideoTePose:
    def __init__(self, hmr, model, model_vibe=None, J_regressor=None, batch=1, use_graph=True):
        nv.require_cuda(next(hmr.parameters()), "HMR parameters")
        self.hmr, self.B = hmr, batch
        self.window = WindowedTePose(model, model_vibe, J_regressor=J_regressor, batch=batch, use_graph=use_graph)
        self.device, self.T = self.window.device, self.window.T
        self.use_graph = use_graph
        self.table = torch.zeros(batch, CROP_FIELDS, dtype=torch.int32, device=self.device)
        self.x4 = torch.zeros(batch, CROP, CROP, 4, dtype=torch.bfloat16, device=self.device)
        self.frames = None                            # [F,H,W,3] uint8, allocated by the first push
        self.pushed = 0
        self.bootstrapped = False                     # VIBE has run on this clip
        self._graph = None
        self._out = None
        self.launches_per_replay = None

    def reset(self):
        """Start a new clip: empty window, unseeded theta ring, VIBE to run again (the captured graph and buffers stay)."""
        self.window.x.zero_()
        self.window.seeded = False
        self.pushed = 0
        self.bootstrapped = False

    def set_theta(self, theta_input: torch.Tensor):
        """Seed the theta ring [B,T-1,85] or [T-1,85] before the T-th push instead of with VIBE's thetas (evaluate.py:219)."""
        self.window.set_theta(theta_input)

    # ------------------------------------------------------------------ one frame
    def _load(self, frames: torch.Tensor, crops):
        if frames.dim() != 4 or frames.shape[3] != 3 or frames.dtype != torch.uint8:
            raise ValueError(f"expected uint8 frames [F,H,W,3], got {tuple(frames.shape)} {frames.dtype}")
        if self.frames is None:
            self.frames = torch.empty(frames.shape, dtype=torch.uint8, device=self.device)
        elif self.frames.shape != frames.shape:
            raise ValueError(f"frames changed shape from {tuple(self.frames.shape)} to {tuple(frames.shape)}; "
                             "use a new VideoTePose per frame size")
        on_device = torch.is_tensor(crops) and crops.is_cuda
        t = crops if on_device else torch.as_tensor(crops, dtype=torch.float64)
        if tuple(t.shape) != (self.B, CROP_FIELDS):
            raise ValueError(f"expected crops [{self.B},{CROP_FIELDS}], got {tuple(t.shape)}")
        if not on_device and not bool(((t[:, 0] >= 0) & (t[:, 0] < frames.shape[0])).all()):
            raise ValueError(f"crop frame indices must lie in [0, {frames.shape[0]})")
        # a host table is pageable: the copy stages it before returning, so the next push cannot overwrite it in flight
        self.table.copy_(make_crop_table(t, t.device), non_blocking=True)
        self.frames.copy_(frames, non_blocking=True)

    def _extract(self):
        """crop -> HMR -> the newest frame of the feature ring"""
        F, H, W, _ = self.frames.shape
        nv.check(nv.lib().tp_crop_normalize_bf16(nv.ptr(self.frames), F, H, W, nv.ptr(self.table), self.B, nv.ptr(self.x4),
                                                 nv.stream()), "tp_crop_normalize_bf16")
        self.window.push_features(self.hmr.features_nhwc4(self.x4))

    def _steady(self):
        self._extract()
        return self.window._body()

    @torch.no_grad()
    @nv.device_guard
    def push(self, frames: torch.Tensor, crops):
        """frames uint8 [F,H,W,3] RGB (CUDA or pinned host); crops [B,6] rows (frame, cx, cy, w, h, scale) with frame indexing
        `frames` (host or CUDA).  Returns None for the first T-1 pushes; at the T-th, VIBE's outputs
        for frames 0..T-2 followed by the first window's, [B,T,...] each; afterwards the newest frame's outputs, [B,...] each
        (tensors reused by the next push when graphs are on)."""
        self._load(frames, crops)
        self.pushed += 1
        if self.pushed < self.T:
            self._extract()
            return None
        if self.pushed == self.T:
            self._extract()
            win = self.window
            first = None
            if not self.bootstrapped:
                if win.vibe is None and not win.seeded:
                    raise RuntimeError("VideoTePose was built without a bootstrap model: call set_theta() before the T-th push")
                if win.vibe is not None:
                    first = win.bootstrap(win.features.clone(), seed_ring=not win.seeded)
                self.bootstrapped = True
            out = win._body()
            if first is None:
                return {k: out[k][:, None] for k in out}
            return {k: torch.cat([first[k], out[k][:, None]], 1) for k in out if k in first}
        if not self.use_graph:
            return self._steady()
        if self._graph is None:
            self._graph, self._out, self.launches_per_replay = self.window._capture(self._steady)
        self._graph.replay()
        return self._out

    # ------------------------------------------------------------------ whole clip
    @torch.no_grad()
    def run(self, frames: torch.Tensor, crops, theta_input=None, keys=OUTPUT_KEYS, bootstrap_frames=None):
        """frames uint8 [N,H,W,3] (or [N,F,H,W,3]: F frames per time step), crops [B,N,6]: row crops[b, t] crops frame t
        (frame field 0, or an index into the F frames of step t).  Returns {key: [B,N,...]} as WindowedTePose.run does on the
        features HMR extracts from those crops: frames 0..T-2 from the bootstrap model, frame k+T-1 from window k.
        theta_input seeds the ring instead of VIBE's thetas; bootstrap_frames: how many frames VIBE sees (default T; the
        demo passes N, whose features are then extracted once more, eagerly, before the window loop)."""
        B, T = self.B, self.T
        if frames.dim() == 4:
            frames = frames[:, None]
        crops = torch.as_tensor(crops) if not torch.is_tensor(crops) else crops
        N = frames.shape[0]
        if frames.dim() != 5 or N < T or tuple(crops.shape) != (B, N, CROP_FIELDS):
            raise ValueError(f"expected frames [N>={T},(F,)H,W,3] and crops [{B},N,{CROP_FIELDS}], got {tuple(frames.shape)}, "
                             f"{tuple(crops.shape)}")
        self.reset()
        nb = T if bootstrap_frames is None else int(bootstrap_frames)
        if not T <= nb <= N:
            raise ValueError(f"bootstrap_frames must lie in [{T}, {N}], got {nb}")
        if theta_input is not None:
            self.set_theta(theta_input)
        res = None
        if nb > T:                                      # VIBE over more than the first window: its features first
            feats = torch.stack([self.hmr.features_from_frames(frames[t].to(self.device), crops[:, t]) for t in range(nb)], 1)
            first = self.window.bootstrap(feats, seed_ring=theta_input is None)
            self.bootstrapped = True
            res = {k: torch.empty((B, N) + tuple(first[k].shape[2:]), device=self.device) for k in keys}
            for k in keys:
                res[k][:, :T - 1].copy_(first[k])
            for t in range(T):
                out = self.push(frames[t], crops[:, t])
            for k in keys:
                res[k][:, T - 1].copy_(out[k][:, -1])
        else:
            for t in range(T):
                out = self.push(frames[t], crops[:, t])
            res = {k: torch.empty((B, N) + tuple(out[k].shape[2:]), device=self.device) for k in keys}
            for k in keys:
                res[k][:, :T].copy_(out[k])
        for t in range(T, N):
            out = self.push(frames[t], crops[:, t])
            for k in keys:
                res[k][:, t].copy_(out[k])
        return res
