"""The windowed loop per tracked person, for tracker output where people enter, leave and are missed for a few frames.

The reference demo treats every tracked person as a sequence of its own (demo.py:183-252): the person's frames, the person's
VIBE bootstrap, then the sliding T-frame window over those frames.  Here S *slots* share one WindowedTePose of batch S: slot s
holds row s of the window state x [S,T,2133] (features | theta ring) and follows one track at a time.  A push hands the
kernels a device table of S entries (tp_window_slots_push / tp_window_slots_commit, include/tepose_b200.h):

    op[s]   0 = no frame for slot s this push, 1 = the next frame of its track, 2 = the first frame of a new track
    src[s]  the row of this push's feature batch that belongs to slot s

so one captured graph follows tracks as they start, pause and end.  A push is

    slot push kernel (graph) -> [VIBE at batch S over the whole window, only when a track reaches its T-th frame]
                             -> window step at batch S + commit kernel (graph)

A track has no output before its T-th frame; at its T-th it returns VIBE's frames 0..T-2 and the first window's frame (VIBE
runs at batch S, so its row sees the kernels WindowedTePose.run uses; only the bootstrapping slots' rings are seeded); after
that one frame per push.  A track absent from a push keeps its slot, its window and its ring (op 0), as in the demo, where a
track is the list of its own frames; end() / end_missing() free the slot.

TrackedVideoTePose puts the crop and the HMR trunk in front, for the n people present only: the crop table is compacted to
those n rows and the trunk runs at the next power of two >= n (capped at S), one captured graph per size.

    tt = TrackedTePose(model, model_vibe, J_regressor=J, slots=8)
    out = tt.push(feats [n,2048], track_ids)        # {track_id: {theta [k,85], verts [k,6890,3], ...}}, k in {1, T}
    tt.end_missing()
  or a whole clip:
    res = tt.run({track_id: (first_frame or frame_ids [n], feats [n,2048])})      # {track_id: {key: [n,...]}}

    tv = TrackedVideoTePose(hmr, model, model_vibe, J_regressor=J, slots=8)
    out = tv.push(frames [F,H,W,3] uint8, {track_id: (frame, cx, cy, w, h, scale)})
    res = tv.run(frames [N,H,W,3], {track_id: (frame_ids [n], boxes [n,5] (cx, cy, w, h, scale))})

The bookkeeping (SlotTable, bucket, compact_crops, schedule) is plain Python and runs without a GPU.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _native as nv
from .hmr import CROP, CROP_FIELDS, make_crop_table
from .stream import FEAT, OUTPUT_KEYS, WindowedTePose

OP_NONE, OP_NEXT, OP_START = 0, 1, 2


# ---------------------------------------------------------------------------------------------------- bookkeeping
class SlotPlan:
    """One push's slot assignment: ids / slots / counts per present track (in push order; `counts` includes this push), and the
    op / src tables of the S slots."""

    def __init__(self, ids, slots, counts, op, src):
        self.ids, self.slots, self.counts, self.op, self.src = ids, slots, counts, op, src


class SlotTable:
    """Which track holds which slot.  A new track takes the lowest free slot (op 2), a known one continues (op 1), and every
    other slot gets op 0; src of a present track is its row in the push."""

    def __init__(self, slots: int):
        if int(slots) < 1:
            raise ValueError(f"slots must be >= 1, got {slots}")
        self.S = int(slots)
        self.slot_of = {}          # track id -> slot
        self.frames = {}           # track id -> frames pushed so far
        self.last = set()          # the ids of the last push
        self.pushes = 0

    def plan(self, track_ids) -> SlotPlan:
        """The assignment of a push of `track_ids`, without applying it.  Raises ValueError for a repeated id or more live tracks
        than slots."""
        ids = list(track_ids)
        if len(set(ids)) != len(ids):
            raise ValueError(f"push {self.pushes}: a track id appears twice in {ids}")
        new = [i for i in ids if i not in self.slot_of]
        free = sorted(set(range(self.S)) - set(self.slot_of.values()))
        if len(new) > len(free):
            raise ValueError(f"push {self.pushes}: {len(self.slot_of) + len(new)} live tracks for {self.S} slots "
                             f"(end() or end_missing() frees the slots of finished tracks)")
        taken = dict(zip(new, free))
        op, src = [OP_NONE] * self.S, [0] * self.S
        slots, counts = [], []
        for row, i in enumerate(ids):
            s = self.slot_of.get(i, taken.get(i))
            op[s] = OP_START if i in taken else OP_NEXT
            src[s] = row
            slots.append(s)
            counts.append(self.frames.get(i, 0) + 1)
        return SlotPlan(ids, slots, counts, op, src)

    def apply(self, plan: SlotPlan) -> None:
        for i, s, c in zip(plan.ids, plan.slots, plan.counts):
            self.slot_of[i], self.frames[i] = s, c
        self.last = set(plan.ids)
        self.pushes += 1

    def end(self, track_id) -> int:
        """Frees the slot of `track_id` and returns it."""
        if track_id not in self.slot_of:
            raise ValueError(f"track {track_id!r} holds no slot")
        del self.frames[track_id]
        return self.slot_of.pop(track_id)

    def end_missing(self):
        """Frees every slot whose track was absent from the last push; returns those track ids."""
        gone = [i for i in self.slot_of if i not in self.last]
        for i in gone:
            self.end(i)
        return gone

    def reset(self) -> None:
        self.slot_of.clear()
        self.frames.clear()
        self.last = set()


def bucket(n: int, slots: int) -> int:
    """The batch the HMR trunk runs at for n people present: the next power of two >= n, capped at `slots`."""
    if not 1 <= n <= slots:
        raise ValueError(f"need 1 <= n <= slots, got n={n}, slots={slots}")
    b = 1
    while b < n:
        b *= 2
    return min(b, slots)


def compact_crops(rows, nb: int) -> np.ndarray:
    """rows [n,6] (frame, cx, cy, w, h, scale) of the people present -> the crop rows [nb,6] of the trunk's batch: the n rows
    first, then copies of row 0 (a valid box; their features are never referenced by src)."""
    r = np.asarray(rows, np.float64).reshape(-1, CROP_FIELDS)
    if not 1 <= r.shape[0] <= nb:
        raise ValueError(f"need 1 <= n <= {nb} crop rows, got {r.shape[0]}")
    return np.concatenate([r, np.repeat(r[:1], nb - r.shape[0], 0)], 0)


def frame_ids(spec, n: int, name) -> np.ndarray:
    """A track's frames: an int (the first frame; the track is then contiguous) or n strictly increasing frame ids >= 0."""
    if np.ndim(spec) == 0:
        f0 = int(spec)
        ids = np.arange(f0, f0 + n)
    else:
        ids = np.asarray(spec)
        if ids.shape != (n,) or not np.issubdtype(ids.dtype, np.integer):
            raise ValueError(f"track {name!r}: expected {n} integer frame ids, got shape {ids.shape} {ids.dtype}")
    if n < 1 or ids[0] < 0 or (n > 1 and not bool((np.diff(ids) > 0).all())):
        raise ValueError(f"track {name!r}: frame ids must be >= 0 and strictly increasing, with at least one frame")
    return ids.astype(np.int64)


def schedule(frames_by_track):
    """{id: frame ids [n]} -> [(frame, [(id, index of that frame in the track)], [ids whose last frame this is])] over the frames
    where someone is present, in increasing order."""
    at = {}
    for i, ids in frames_by_track.items():
        for k, f in enumerate(ids.tolist()):
            at.setdefault(f, []).append((i, k))
    return [(f, at[f], [i for i, k in at[f] if k == len(frames_by_track[i]) - 1]) for f in sorted(at)]


# ---------------------------------------------------------------------------------------------------- features -> meshes
class TrackedTePose:
    def __init__(self, model, model_vibe=None, J_regressor=None, slots=1):
        self.table = SlotTable(slots)
        self.S = self.table.S
        self.window = WindowedTePose(model, model_vibe, J_regressor=J_regressor, batch=self.S)
        self.device, self.T = self.window.device, self.window.T
        self.feats = torch.zeros(self.S, FEAT, device=self.device)                        # this push's features, src rows
        self.tab = torch.zeros(2, self.S, dtype=torch.int32, device=self.device)          # [op; src]
        self.seed = {}                       # slot -> theta_input [T-1,85] given at the track's first push
        self._push_graph = self._step_graph = self._out = None
        self.launches_per_replay = None      # native launches of the push graph + the step graph

    # ------------------------------------------------------------------ slots
    def end(self, track_id) -> None:
        """Frees the slot of a finished track (its window and seed are dropped when the slot's next track starts)."""
        self.table.end(track_id)

    def end_missing(self):
        """Frees every slot whose track was absent from the last push; returns those track ids."""
        return self.table.end_missing()

    def reset(self) -> None:
        """Frees every slot."""
        self.table.reset()
        self.seed.clear()

    # ------------------------------------------------------------------ one push
    def _push_kernel(self):
        S, T = self.S, self.T
        nv.check(nv.lib().tp_window_slots_push(nv.ptr(self.window.x), S, T, FEAT + 85, nv.ptr(self.feats), nv.ptr(self.tab[1]),
                                               nv.ptr(self.tab[0]), nv.stream()), "tp_window_slots_push")

    def _step(self):
        win = self.window
        out = win.model(win.x, J_regressor=win.J_regressor)[-1]
        nv.check(nv.lib().tp_window_slots_commit(nv.ptr(win.x), self.S, self.T, FEAT + 85, nv.ptr(out["theta"].contiguous()),
                                                 nv.ptr(self.tab[0]), nv.stream()), "tp_window_slots_commit")
        return out

    def _seeds(self, plan, theta_input):
        """theta_input {track id: [T-1,85]} for tracks that start at this push -> {slot: device tensor}."""
        seeds = {}
        for i, tin in (theta_input or {}).items():
            if i not in plan.ids or plan.counts[plan.ids.index(i)] != 1:
                raise ValueError(f"push {self.table.pushes}: theta_input for track {i!r}, which does not start at this push")
            t = torch.as_tensor(tin).to(self.device, torch.float32)
            if tuple(t.shape) != (self.T - 1, 85):
                raise ValueError(f"theta_input of track {i!r} must be [{self.T - 1},85], got {tuple(t.shape)}")
            seeds[plan.slots[plan.ids.index(i)]] = t
        if self.window.vibe is None:
            for i, s, c in zip(plan.ids, plan.slots, plan.counts):
                if c == 1 and s not in seeds:
                    raise ValueError(f"push {self.table.pushes}: track {i!r} starts without theta_input and there is no "
                                     "bootstrap model")
        return seeds

    def _advance(self, plan: SlotPlan, seeds):
        """The window work of a push whose features are already in self.feats (row plan.src[s] for slot s); seeds: _seeds()."""
        self.table.apply(plan)
        for s in plan.slots:                 # a slot that starts a track forgets its previous track's seed
            if plan.op[s] == OP_START:
                self.seed.pop(s, None)
        self.seed.update(seeds)
        if not plan.ids:
            return {}
        # a host table is pageable: the copy stages it before returning, so the next push cannot overwrite it in flight
        self.tab.copy_(torch.tensor([plan.op, plan.src], dtype=torch.int32), non_blocking=True)
        win = self.window
        if self._push_graph is None:
            self._push_graph, _, n_push = win._capture(self._push_kernel)
            self._step_graph, self._out, n_step = win._capture(self._step)
            self.launches_per_replay = n_push + n_step
        self._push_graph.replay()
        boot = [s for s, c in zip(plan.slots, plan.counts) if c == self.T]
        first = None
        if boot:
            if win.vibe is not None:
                first = win.bootstrap(win.features.clone(), seed_ring=False)
            for s in boot:
                win.theta_input[s].copy_(self.seed[s] if s in self.seed else first["theta"][s])
        self._step_graph.replay()
        out = self._out
        res = {}
        for i, s, c in zip(plan.ids, plan.slots, plan.counts):
            if c > self.T or (c == self.T and first is None):
                res[i] = {k: out[k][s:s + 1] for k in OUTPUT_KEYS}
            elif c == self.T:
                res[i] = {k: torch.cat([first[k][s], out[k][s:s + 1]], 0) for k in OUTPUT_KEYS}
        return res

    @torch.no_grad()
    @nv.device_guard
    def push(self, feats: torch.Tensor, track_ids, theta_input=None):
        """feats [n,2048] (CUDA or pinned host): the newest frame of each of the n tracks present, in the order of track_ids.
        theta_input {track id: [T-1,85]}: the ring seed of a track starting at this push, instead of VIBE's thetas
        (evaluate.py:219; required for every new track without a bootstrap model).  Returns {track id: {key: [k,...]}} for the
        tracks with output: k = T at a track's T-th frame (VIBE's frames 0..T-2, then the first window's; k = 1 without VIBE),
        k = 1 afterwards.  Steady outputs are views of tensors the next push reuses."""
        ids = list(track_ids)
        if feats.dim() != 2 or feats.shape[1] != FEAT or feats.shape[0] != len(ids):
            raise ValueError(f"expected feats [{len(ids)},{FEAT}] for {len(ids)} track ids, got {tuple(feats.shape)}")
        plan = self.table.plan(ids)
        seeds = self._seeds(plan, theta_input)
        self.feats[:len(ids)].copy_(feats, non_blocking=True)
        return self._advance(plan, seeds)

    # ------------------------------------------------------------------ whole clip
    @torch.no_grad()
    def run(self, features_by_track, theta_input=None, keys=OUTPUT_KEYS):
        """features_by_track {id: (first frame or frame ids [n], feats [n,2048])}: frame ids strictly increasing, gaps meaning
        the person was missed.  Returns {id: {key: [n,...]}} for the tracks with at least T frames: each track's outputs as
        WindowedTePose.run gives them for its own frames (frames 0..T-2 from VIBE; NaN without a bootstrap model).
        theta_input {id: [T-1,85]} seeds those tracks' rings.  Every slot is freed first, and each track after its last frame."""
        frames, feats = {}, {}
        for i, (spec, f) in features_by_track.items():
            f = torch.as_tensor(f)
            if f.dim() != 2 or f.shape[1] != FEAT or f.shape[0] < 1:
                raise ValueError(f"track {i!r}: expected feats [n>=1,{FEAT}], got {tuple(f.shape)}")
            frames[i], feats[i] = frame_ids(spec, f.shape[0], i), f.to(self.device, torch.float32)
        return _run_clip(self, frames, lambda f, present, tin: self.push(
            torch.stack([feats[i][k] for i, k in present]), [i for i, _ in present], tin), theta_input, keys)


def _run_clip(owner, frames, push, theta_input, keys):
    """The per-person loop of a whole clip: frames {id: frame ids [n]}; push(frame, [(id, index)], theta_input) -> the push's
    outputs.  Returns {id: {key: [n,...]}}."""
    unknown = set(theta_input or {}) - set(frames)
    if unknown:
        raise ValueError(f"theta_input for unknown tracks {sorted(map(repr, unknown))}")
    owner.reset()
    res = {}
    for f, present, ending in schedule(frames):
        tin = {i: theta_input[i] for i, k in present if k == 0 and i in (theta_input or {})}
        out = push(f, present, tin or None)
        for i, k in present:
            if i not in out:
                continue
            if i not in res:
                res[i] = {key: torch.full((len(frames[i]),) + tuple(out[i][key].shape[1:]), float("nan"), device=owner.device)
                          for key in keys}
            m = out[i][keys[0]].shape[0]                # T at the track's T-th frame (with VIBE), else 1
            for key in keys:
                res[i][key][k + 1 - m:k + 1].copy_(out[i][key])
        for i in ending:
            owner.end(i)
    return res


# ---------------------------------------------------------------------------------------------------- frames -> meshes
class TrackedVideoTePose:
    def __init__(self, hmr, model, model_vibe=None, J_regressor=None, slots=1):
        nv.require_cuda(next(hmr.parameters()), "HMR parameters")
        self.hmr = hmr
        self.tracker = TrackedTePose(model, model_vibe, J_regressor=J_regressor, slots=slots)
        self.device, self.T, self.S = self.tracker.device, self.tracker.T, self.tracker.S
        self.frames = None                   # [F,H,W,3] uint8, allocated by the first push
        self.buckets = {}                    # trunk batch -> {table, extract, graph, launches}

    def end(self, track_id) -> None:
        self.tracker.end(track_id)

    def end_missing(self):
        return self.tracker.end_missing()

    def reset(self) -> None:
        self.tracker.reset()

    def _bucket(self, nb):
        """Crop + trunk at batch nb, its features landing in rows 0..nb-1 of the tracker's feature batch (captured at first use)."""
        if nb not in self.buckets:
            split = self.hmr.precision == "fp32_tc"
            table = torch.zeros(nb, CROP_FIELDS, dtype=torch.int32, device=self.device)
            x = torch.zeros(nb, CROP, CROP, self.hmr.stem_channels, dtype=torch.bfloat16, device=self.device)
            name = "tp_crop_normalize_split3" if split else "tp_crop_normalize_bf16"

            def extract():
                F, H, W, _ = self.frames.shape
                nv.check(getattr(nv.lib(), name)(nv.ptr(self.frames), F, H, W, nv.ptr(table), nb, nv.ptr(x), nv.stream()), name)
                self.tracker.feats[:nb].copy_(self.hmr.features_nhwc12(x) if split else self.hmr.features_nhwc4(x))
            self.buckets[nb] = {"table": table, "extract": extract, "graph": None, "launches": None}
        return self.buckets[nb]

    @torch.no_grad()
    @nv.device_guard
    def push(self, frames: torch.Tensor, boxes, theta_input=None):
        """frames uint8 [F,H,W,3] RGB (CUDA or pinned host); boxes {track id: (frame, cx, cy, w, h, scale)} of the people present,
        `frame` indexing `frames`.  Crop and HMR run for those people only, at the trunk batch bucket(n, S).  Returns what
        TrackedTePose.push returns."""
        if frames.dim() != 4 or frames.shape[3] != 3 or frames.dtype != torch.uint8:
            raise ValueError(f"expected uint8 frames [F,H,W,3], got {tuple(frames.shape)} {frames.dtype}")
        if self.frames is not None and self.frames.shape != frames.shape:
            raise ValueError(f"frames changed shape from {tuple(self.frames.shape)} to {tuple(frames.shape)}; "
                             "use a new TrackedVideoTePose per frame size")
        ids = list(boxes)
        plan = self.tracker.table.plan(ids)
        seeds = self.tracker._seeds(plan, theta_input)
        if ids:
            rows = np.array([np.asarray(boxes[i], np.float64).reshape(-1) for i in ids])
            if rows.shape != (len(ids), CROP_FIELDS):
                raise ValueError(f"each box must be (frame, cx, cy, w, h, scale), got rows of shape {rows.shape}")
            if not bool(((rows[:, 0] >= 0) & (rows[:, 0] < frames.shape[0]) & (rows[:, 0] == np.round(rows[:, 0]))).all()):
                raise ValueError(f"box frame indices must be integers in [0, {frames.shape[0]})")
            if self.frames is None:
                self.frames = torch.empty(frames.shape, dtype=torch.uint8, device=self.device)
            nb = bucket(len(ids), self.S)
            b = self._bucket(nb)
            # pageable host table: the copy stages it before returning, so the next push cannot overwrite it in flight
            b["table"].copy_(make_crop_table(compact_crops(rows, nb), "cpu"), non_blocking=True)
            self.frames.copy_(frames, non_blocking=True)
            if b["graph"] is None:
                b["graph"], _, b["launches"] = self.tracker.window._capture(b["extract"])
            b["graph"].replay()
        return self.tracker._advance(plan, seeds)

    @torch.no_grad()
    def run(self, frames: torch.Tensor, tracks, theta_input=None, keys=OUTPUT_KEYS):
        """frames uint8 [N,H,W,3]; tracks {id: (frame ids [n], boxes [n,5] rows (cx, cy, w, h, scale))}, frame ids strictly
        increasing in [0, N) (gaps: the person was missed).  Returns {id: {key: [n,...]}} as TrackedTePose.run does on the
        features of those crops."""
        if frames.dim() != 4 or frames.shape[3] != 3 or frames.dtype != torch.uint8:
            raise ValueError(f"expected uint8 frames [N,H,W,3], got {tuple(frames.shape)} {frames.dtype}")
        N = frames.shape[0]
        ids_of, boxes_of = {}, {}
        for i, (spec, b) in tracks.items():
            b = np.asarray(b.cpu() if torch.is_tensor(b) else b, np.float64)
            if b.ndim != 2 or b.shape[1] != 5:
                raise ValueError(f"track {i!r}: expected boxes [n,5] (cx, cy, w, h, scale), got {b.shape}")
            f = frame_ids(spec, b.shape[0], i)
            if f[-1] >= N:
                raise ValueError(f"track {i!r}: frame {int(f[-1])} of a clip of {N} frames")
            ids_of[i], boxes_of[i] = f, b
        return _run_clip(self, ids_of, lambda f, present, tin: self.push(
            frames[f:f + 1], {i: (0,) + tuple(boxes_of[i][k]) for i, k in present}, tin), theta_input, keys)
