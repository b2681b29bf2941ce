"""The demo's output stage on the device: crop cameras and keypoints in frame coordinates, and every tracked person's mesh drawn
over the frame (lib/utils/demo_utils.py: convert_crop_cam_to_orig_img, convert_crop_coords_to_orig_img; lib/utils/renderer.py:
Renderer.render, called once per person present, each over the previous result).

    r = MeshRenderer(smpl.faces, H, W)
    img = r.render(frame [H,W,3] uint8, verts [n,6890,3], crop_cam_to_frame(theta[:, :3], boxes, W, H))
    video = render_clip(r, frames, tracks, TrackedVideoTePose(...).run(frames, tracks))

The renderer is tp_render_meshes (csrc/render.cu); its contract (projection, fill rule, visibility, shading) is stated in
include/tepose_b200.h and restated in oracle/render_ref.py.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _native as nv
from .tracks import frame_ids

DEFAULT_COLOR = (1.0, 1.0, 0.9)      # lib/utils/renderer.py: Renderer.render's default mesh colour


def _boxes(boxes, like: torch.Tensor) -> torch.Tensor:
    b = torch.as_tensor(boxes).to(like.device, like.dtype)
    if b.dim() != 2 or b.shape[1] != 5:
        raise ValueError(f"expected boxes [n,5] (cx, cy, w, h, scale), got {tuple(b.shape)}")
    return b


def crop_cam_to_frame(cam: torch.Tensor, boxes, width: float, height: float) -> torch.Tensor:
    """cam [n,3] = theta[:, :3] (s, tx, ty) of crops boxes [n,5] (cx, cy, w, h, scale) -> orig_cam [n,4] (sx, sy, tx, ty): the
    weak-perspective camera of the whole width x height frame that puts each point where the crop camera puts it inside the crop,
    which covers w*scale x h*scale frame pixels around (cx, cy) (oracle/crop_ref.py: patch_points):
        sx = s*w*scale/W,  sy = s*h*scale/H,  tx' = tx + (cx - W/2)/(W/2)/sx,  ty' = ty + (cy - H/2)/(H/2)/sy.
    For a square box this is the reference's convert_crop_cam_to_orig_img with bbox[:, 2] equal to the crop side w*scale.  The
    reference demo passes the tracker's box side there (bbox[:, 2] = h, without the crop's scale factor), so at scale != 1 its
    overlay is that factor smaller than what the crop camera saw; this helper follows the crop."""
    if cam.dim() != 2 or cam.shape[1] != 3:
        raise ValueError(f"expected cam [n,3] (s, tx, ty), got {tuple(cam.shape)}")
    b = _boxes(boxes, cam)
    if b.shape[0] != cam.shape[0]:
        raise ValueError(f"{cam.shape[0]} cameras for {b.shape[0]} boxes")
    s, tx, ty = cam.unbind(1)
    cx, cy, w, h, sc = b.unbind(1)
    hw, hh = width / 2.0, height / 2.0
    sx = s * w * sc / width
    sy = s * h * sc / height
    return torch.stack([sx, sy, tx + (cx - hw) / hw / sx, ty + (cy - hh) / hh / sy], 1)


def crop_kp_to_frame(kp_2d: torch.Tensor, boxes) -> torch.Tensor:
    """kp_2d [n,J,2] in the crop's normalised coordinates ([-1, 1] across the crop) -> frame pixels [n,J,2]: the demo's
    joints2d_img_coordinates (convert_crop_coords_to_orig_img) for crops covering w*scale x h*scale pixels around (cx, cy)."""
    if kp_2d.dim() != 3 or kp_2d.shape[2] != 2:
        raise ValueError(f"expected kp_2d [n,J,2], got {tuple(kp_2d.shape)}")
    b = _boxes(boxes, kp_2d)
    if b.shape[0] != kp_2d.shape[0]:
        raise ValueError(f"{kp_2d.shape[0]} keypoint sets for {b.shape[0]} boxes")
    half = torch.stack([b[:, 2] * b[:, 4], b[:, 3] * b[:, 4]], 1)[:, None] / 2
    return b[:, None, :2] + kp_2d * half


def vertex_faces(faces: np.ndarray, num_verts: int):
    """The vertex -> face CSR of faces [F,3]: offsets [V+1] and face ids, each vertex's faces in ascending order (a face that
    repeats a vertex is listed once per corner)."""
    f = np.asarray(faces, np.int64)
    corner_v = f.reshape(-1)
    corner_f = np.repeat(np.arange(f.shape[0]), 3)
    order = np.lexsort((corner_f, corner_v))
    offsets = np.zeros(num_verts + 1, np.int64)
    np.add.at(offsets, corner_v + 1, 1)
    return np.cumsum(offsets).astype(np.int32), corner_f[order].astype(np.int32)


class MeshRenderer:
    """Draws meshes of one topology (faces [F,3], vertex ids in [0, num_verts)) over height x width frames on a CUDA device."""

    def __init__(self, faces, height: int, width: int, num_verts: int = 6890, device="cuda"):
        f = np.asarray(faces.cpu() if torch.is_tensor(faces) else faces)
        if f.ndim != 2 or f.shape[1] != 3 or not np.issubdtype(f.dtype, np.integer):
            raise ValueError(f"expected integer faces [F,3], got {f.shape} {f.dtype}")
        if not 1 <= f.shape[0] <= 65536:
            raise ValueError(f"need 1 <= F <= 65536 faces, got {f.shape[0]}")
        if f.min() < 0 or f.max() >= num_verts:
            raise ValueError(f"face vertex ids must lie in [0, {num_verts}), got [{f.min()}, {f.max()}]")
        if not (1 <= int(height) <= 32768 and 1 <= int(width) <= 32768):
            raise ValueError(f"need 1 <= height, width <= 32768, got {height} x {width}")
        self.device = torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        nv.require_cuda(torch.empty(0, device=self.device), "MeshRenderer device")
        self.H, self.W, self.V, self.F = int(height), int(width), int(num_verts), int(f.shape[0])
        off, ids = vertex_faces(f, self.V)
        self.faces = torch.from_numpy(f.astype(np.int32)).to(self.device)
        self.vf_offsets = torch.from_numpy(off).to(self.device)
        self.vf_faces = torch.from_numpy(ids).to(self.device)
        self._ws = None

    def _workspace(self, n):
        need = nv.lib().tp_render_workspace_bytes(n, self.V, self.H, self.W)
        if self._ws is None or self._ws.numel() < need:
            self._ws = nv.workspace(need, self.device)
        return self._ws

    @torch.no_grad()
    @nv.device_guard
    def render(self, frame: torch.Tensor, verts: torch.Tensor, orig_cam: torch.Tensor, colors=None) -> torch.Tensor:
        """frame uint8 [H,W,3]; verts [n,V,3], orig_cam [n,4] (crop_cam_to_frame), colors [n,3] in [0,1] (default
        DEFAULT_COLOR) -> a new uint8 [H,W,3] CUDA tensor: person n-1 over person n-2 ... over person 0 over the frame."""
        for name, t in (("frame", frame), ("verts", verts), ("orig_cam", orig_cam)):
            nv.require_cuda(t, name)
            if t.device != self.device:
                raise ValueError(f"{name} is on {t.device}, the renderer on {self.device}")
        if frame.dtype != torch.uint8 or tuple(frame.shape) != (self.H, self.W, 3):
            raise ValueError(f"expected uint8 frame [{self.H},{self.W},3], got {tuple(frame.shape)} {frame.dtype}")
        n = verts.shape[0] if verts.dim() == 3 else -1
        if verts.dim() != 3 or tuple(verts.shape[1:]) != (self.V, 3):
            raise ValueError(f"expected verts [n,{self.V},3], got {tuple(verts.shape)}")
        if tuple(orig_cam.shape) != (n, 4):
            raise ValueError(f"expected orig_cam [{n},4], got {tuple(orig_cam.shape)}")
        if n > 65535:
            raise ValueError(f"at most 65535 people per frame, got {n}")
        if colors is None:
            colors = torch.tensor(DEFAULT_COLOR, dtype=torch.float32, device=self.device).expand(n, 3)
        colors = torch.as_tensor(colors, dtype=torch.float32).to(self.device)
        if tuple(colors.shape) != (n, 3):
            raise ValueError(f"expected colors [{n},3], got {tuple(colors.shape)}")
        frame = frame.contiguous()
        verts = verts.to(torch.float32).contiguous()
        cam = orig_cam.to(torch.float32).contiguous()
        colors = colors.contiguous()
        out = torch.empty_like(frame)
        ws = self._workspace(n)
        nv.check(nv.lib().tp_render_meshes(nv.ptr(frame), nv.ptr(verts), nv.ptr(cam), nv.ptr(colors), nv.ptr(self.faces),
                                           nv.ptr(self.vf_offsets), nv.ptr(self.vf_faces), n, self.V, self.F, self.H, self.W,
                                           nv.ptr(out), nv.ptr(ws), ws.numel(), nv.stream()), "tp_render_meshes")
        return out


@torch.no_grad()
def render_clip(renderer: MeshRenderer, frames: torch.Tensor, tracks, results, colors=None) -> torch.Tensor:
    """frames uint8 [N,H,W,3]; tracks {id: (frame ids, boxes [n,5])} and results {id: {"theta", "verts", ...}} as given to and
    returned by TrackedVideoTePose.run; colors {id: (r, g, b)} (default DEFAULT_COLOR).  Returns uint8 [N,H,W,3] on the
    renderer's device: in every frame, each track with output there, drawn in the order of `tracks` with its own camera
    (crop_cam_to_frame).  Rows a track has no output for (NaN) draw nothing."""
    if frames.dim() != 4 or frames.shape[3] != 3 or frames.dtype != torch.uint8:
        raise ValueError(f"expected uint8 frames [N,H,W,3], got {tuple(frames.shape)} {frames.dtype}")
    frames = frames.to(renderer.device)
    N = frames.shape[0]
    at = [[] for _ in range(N)]                  # frame -> [(id, row)] in the order of tracks
    for i, (spec, boxes) in tracks.items():
        if i not in results:
            continue
        b = np.asarray(boxes.cpu() if torch.is_tensor(boxes) else boxes, np.float64)
        f = frame_ids(spec, b.shape[0], i)
        if f[-1] >= N:
            raise ValueError(f"track {i!r}: frame {int(f[-1])} of a clip of {N} frames")
        for k, fr in enumerate(f.tolist()):
            at[fr].append((i, k))
    cams = {}
    for i, (spec, boxes) in tracks.items():
        if i in results:
            th = results[i]["theta"].to(renderer.device, torch.float32)
            cams[i] = crop_cam_to_frame(th[:, :3], torch.as_tensor(np.asarray(
                boxes.cpu() if torch.is_tensor(boxes) else boxes, np.float64)), renderer.W, renderer.H)
    out = torch.empty_like(frames)
    for fr in range(N):
        present = at[fr]
        if not present:
            out[fr].copy_(frames[fr])
            continue
        verts = torch.stack([results[i]["verts"][k] for i, k in present])
        cam = torch.stack([cams[i][k] for i, k in present])
        col = None if colors is None else [colors.get(i, DEFAULT_COLOR) for i, _ in present]
        out[fr].copy_(renderer.render(frames[fr], verts, cam, col))
    return out
