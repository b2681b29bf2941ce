"""The reference's live loop kept on the device -- evaluate.py:229-269 / demo.py:229-252, SURVEY.md 8(f-1).

Per sequence the reference (i) runs the VIBE bootstrap model on the first T frames and reports its
first T-1 frames, (ii) for every later frame assembles a [1,T,2133] window on the host -- T static
features, the T-1 most recent predicted thetas, zeros in the newest frame's theta slot -- runs TePose
on it from h0 = 0, copies every output to the host and rolls the theta buffer.  Here the window, the
theta ring and the roll live in HBM, one frame is one CUDA-graph replay, and B independent streams
advance side by side.  The arithmetic per window is exactly TePose.forward (this is NOT the O(N)
carried-state mode of live.py, which is a different function of the stream).

    ws = WindowedTePose(model, model_vibe, J_regressor=J, batch=1)
    out = ws.run(features)                 # features [B,N,2048] -> {theta [B,N,85], verts [B,N,6890,3], ...}
  or frame by frame:
    first = ws.bootstrap(features[:, :T])  # VIBE: frames 0..T-2; seeds the theta ring (demo.py:237)
    out_t = ws.step(features[:, k:k+T])    # frame k+T-1
"""
from __future__ import annotations

import torch

from . import _native as nv

FEAT = 2048
OUTPUT_KEYS = ("theta", "verts", "kp_2d", "kp_3d", "rotmat")


class WindowedTePose:
    def __init__(self, model, model_vibe=None, J_regressor=None, batch=1, use_graph=True):
        p = next(model.parameters())
        nv.require_cuda(p, "model parameters")
        self.model, self.vibe, self.device, self.B = model, model_vibe, p.device, batch
        self.T = int(model.seqlen)
        if self.T < 2:
            raise ValueError("the windowed loop needs seqlen >= 2")
        self.J_regressor = None if J_regressor is None else J_regressor.to(self.device)
        self.x = torch.zeros(batch, self.T, FEAT + 85, device=self.device)      # the window, theta slots included
        self.use_graph = use_graph
        self._graph = None
        self._out = None
        self.launches_per_replay = None
        self.seeded = False

    # ------------------------------------------------------------------ theta ring
    @property
    def theta_input(self):
        """[B,T-1,85] view: the thetas fed to the next window (evaluate.py:252)."""
        return self.x[:, :self.T - 1, FEAT:]

    def set_theta(self, theta_input: torch.Tensor):
        """Seed the ring with given thetas [B,T-1,85] or [T-1,85] (evaluate.py:219 uses the dataset's pseudo thetas)."""
        t = theta_input.to(self.device, torch.float32)
        self.theta_input.copy_(t.reshape(-1, self.T - 1, 85).expand(self.B, -1, -1))
        self.seeded = True

    @torch.no_grad()
    def bootstrap(self, feats: torch.Tensor, seed_ring=True):
        """VIBE over feats [B,>=T,2048] (evaluate.py:233-234 passes the first T frames, demo.py:229 the whole
        clip).  Returns VIBE's outputs for the first T-1 frames and (seed_ring) feeds its thetas to the ring
        (demo.py:237)."""
        if self.vibe is None:
            raise RuntimeError("WindowedTePose was built without a bootstrap model; use set_theta()")
        feats = feats.to(self.device, torch.float32)
        out = self.vibe(feats, J_regressor=self.J_regressor)[-1]
        first = {k: v[:, :self.T - 1] for k, v in out.items()}
        if seed_ring:
            self.theta_input.copy_(first["theta"])
            self.seeded = True
        return first

    # ------------------------------------------------------------------ one frame
    def _body(self):
        T = self.T
        out = self.model(self.x, J_regressor=self.J_regressor)[-1]
        th = self.x[:, :, FEAT:]
        if T > 2:
            th[:, :T - 2].copy_(th[:, 1:T - 1].clone())        # evaluate.py:268
        th[:, T - 2].copy_(out["theta"])                        # evaluate.py:269
        return out

    @torch.no_grad()
    @nv.device_guard
    def step(self, window_feats: torch.Tensor):
        """window_feats [B,T,2048] (CUDA or pinned host): the static features of the T newest frames.
        Returns the prediction for the newest one (tensors are reused by the next call when graphs are on)."""
        if not self.seeded:
            raise RuntimeError("theta ring is not seeded: call bootstrap() or set_theta() first")
        if tuple(window_feats.shape) != (self.B, self.T, FEAT):
            raise ValueError(f"expected window features [{self.B},{self.T},{FEAT}], got {tuple(window_feats.shape)}")
        self.x[:, :, :FEAT].copy_(window_feats, non_blocking=True)
        if not self.use_graph:
            return self._body()
        if self._graph is None:
            self._graph, self._out, self.launches_per_replay = self._capture(self._body)
        self._graph.replay()
        return self._out

    def _capture(self, fn):
        """fn (which advances the rings in self.x) as a CUDA graph: one warm-up run on a side stream (packs weights, sets kernel
        attributes), then the capture; the window is restored after each.  Returns (graph, fn's static output, native kernel
        launches per replay)."""
        keep = self.x.clone()
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            fn()
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        self.x.copy_(keep)
        graph = torch.cuda.CUDAGraph()
        before = nv.lib().tp_launch_count()
        with torch.cuda.graph(graph):
            out = fn()
        launches = int(nv.lib().tp_launch_count() - before)
        self.x.copy_(keep)
        return graph, out, launches

    # ------------------------------------------------------------------ feature ring (tepose_b200.video)
    @property
    def features(self):
        """[B,T,2048] view: the static features of the window, oldest frame first."""
        return self.x[:, :, :FEAT]

    def push_features(self, feats: torch.Tensor):
        """Shift the feature ring by one frame: feats [B,2048] (on the device) becomes the newest frame of the window."""
        f = self.features
        f[:, :self.T - 1].copy_(f[:, 1:].clone())
        f[:, self.T - 1].copy_(feats)

    # ------------------------------------------------------------------ whole sequence
    @torch.no_grad()
    def run(self, features: torch.Tensor, theta_input=None, keys=OUTPUT_KEYS, bootstrap_frames=None):
        """features [B,N,2048], N >= T.  Frames 0..T-2 come from the bootstrap model, frame k+T-1 from window k
        (evaluate.py:233-269).  theta_input, if given, seeds the ring instead of VIBE's thetas (evaluate.py:219).
        bootstrap_frames: how many frames VIBE sees (default T, evaluate.py:233; demo.py:229 passes N)."""
        B, T = self.B, self.T
        if features.dim() != 3 or features.shape[0] != B or features.shape[2] != FEAT or features.shape[1] < T:
            raise ValueError(f"expected features [{B},N>={T},{FEAT}], got {tuple(features.shape)}")
        feats = features.to(self.device, torch.float32)
        N = feats.shape[1]
        nb = T if bootstrap_frames is None else int(bootstrap_frames)
        first = self.bootstrap(feats[:, :nb], seed_ring=theta_input is None)
        if theta_input is not None:
            self.set_theta(theta_input)
        res = {}
        for k in keys:
            res[k] = torch.empty((B, N) + tuple(first[k].shape[2:]), device=self.device, dtype=torch.float32)
            res[k][:, :T - 1].copy_(first[k])
        for i in range(N - T + 1):
            out = self.step(feats[:, i:i + T])
            for k in keys:
                res[k][:, i + T - 1].copy_(out[k])
        return res
