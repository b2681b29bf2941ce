"""Per-track windowed loop (tepose_b200.tracks).  CPU: the slot bookkeeping and the input checks of both run()s.  GPU: the two
slot kernels bit for bit against a torch restatement, TrackedTePose.run against WindowedTePose.run per track, and
TrackedVideoTePose.run against TrackedTePose.run on the features HMR extracts from the same compacted crops."""
import ctypes

import numpy as np
import pytest
import torch

from tepose_b200.tracks import (OP_NEXT, OP_NONE, OP_START, SlotTable, TrackedTePose, TrackedVideoTePose, bucket,
                                compact_crops, frame_ids, schedule)

DEV = "cuda:0"
SEED = 71
KEYS = ("theta", "verts", "kp_2d", "kp_3d", "rotmat")
COLS = 2048 + 85


# ------------------------------------------------------------------------------------------------ CPU: bookkeeping
def test_slot_assignment_and_reuse():
    t = SlotTable(3)
    p = t.plan(["a", "b"])
    assert p.slots == [0, 1] and p.op == [OP_START, OP_START, OP_NONE] and p.src == [0, 1, 0] and p.counts == [1, 1]
    t.apply(p)
    p = t.plan(["c", "b"])                       # b continues, c takes the lowest free slot, a is absent
    assert p.slots == [2, 1] and p.op == [OP_NONE, OP_NEXT, OP_START] and p.src == [0, 1, 0] and p.counts == [1, 2]
    t.apply(p)
    p = t.plan(["a"])                            # a missed for one push: same slot, its next frame
    assert p.slots == [0] and p.op == [OP_NEXT, OP_NONE, OP_NONE] and p.counts == [2]
    t.apply(p)
    assert t.end("b") == 1
    p = t.plan(["d", "a"])                       # b's slot goes to the next new track
    assert p.slots == [1, 0] and p.op == [OP_NEXT, OP_START, OP_NONE] and p.src == [1, 0, 0]
    t.apply(p)
    assert sorted(t.end_missing()) == ["c"]      # absent from the last push
    assert t.slot_of == {"a": 0, "d": 1}
    p = t.plan(["b"])                            # an ended id that comes back is a new track
    assert p.op[2] == OP_START and p.counts == [1]


def test_more_tracks_than_slots_names_the_push_and_changes_nothing():
    t = SlotTable(2)
    t.apply(t.plan([1, 2]))
    t.apply(t.plan([1]))
    before = (dict(t.slot_of), dict(t.frames), t.pushes)
    with pytest.raises(ValueError, match="push 2: 3 live tracks for 2 slots"):
        t.plan([1, 3])                           # 2 is absent but still holds its slot
    assert (dict(t.slot_of), dict(t.frames), t.pushes) == before
    with pytest.raises(ValueError, match="twice"):
        t.plan([1, 1])
    t.end_missing()
    assert t.plan([1, 3]).slots == [0, 1]
    with pytest.raises(ValueError):
        SlotTable(0)
    with pytest.raises(ValueError):
        t.end(7)


def test_lifecycle_tables():
    """start, continue, missing, end + reuse, short track: op per slot and the frame count of each track over a schedule."""
    frames = {"long": np.arange(0, 8), "gap": np.array([0, 1, 4, 5]), "short": np.array([1, 2]), "late": np.arange(3, 8)}
    t = SlotTable(3)
    ops, counts = [], {}
    for f, present, ending in schedule(frames):
        p = t.plan([i for i, _ in present])
        t.apply(p)
        ops.append(p.op)
        for i, c in zip(p.ids, p.counts):
            counts.setdefault(i, []).append(c)
        for i in ending:
            t.end(i)
    assert [f for f, _, _ in schedule(frames)] == list(range(8))
    assert ops == [[2, 2, 0], [1, 1, 2], [1, 0, 1], [1, 0, 2], [1, 1, 1], [1, 1, 1], [1, 0, 1], [1, 0, 1]]
    assert counts == {"long": list(range(1, 9)), "gap": [1, 2, 3, 4], "short": [1, 2], "late": list(range(1, 6))}
    assert t.slot_of == {}


def test_bucket_and_compaction():
    assert [bucket(n, 32) for n in (1, 2, 3, 4, 5, 9, 16, 17, 32)] == [1, 2, 4, 4, 8, 16, 16, 32, 32]
    assert bucket(5, 6) == 6 and bucket(3, 8) == 4 and bucket(1, 1) == 1
    for n, s in ((0, 4), (5, 4)):
        with pytest.raises(ValueError):
            bucket(n, s)
    rows = np.array([(0, 10.0, 20.0, 30.0, 40.0, 1.2), (1, 5.0, 6.0, 7.0, 8.0, 1.0), (0, 1.0, 2.0, 3.0, 4.0, 1.1)])
    c = compact_crops(rows, 4)
    assert c.shape == (4, 6) and np.array_equal(c[:3], rows) and np.array_equal(c[3], rows[0])
    assert np.array_equal(compact_crops(rows, 3), rows)
    with pytest.raises(ValueError):
        compact_crops(rows, 2)


def test_frame_ids():
    assert frame_ids(3, 4, "a").tolist() == [3, 4, 5, 6]
    assert frame_ids([0, 2, 7], 3, "a").tolist() == [0, 2, 7]
    for spec, n in (([0, 2, 2], 3), ([3, 1], 2), ([-1, 0], 2), ([0, 1], 3), (-2, 2), ([0.0, 1.0], 2)):
        with pytest.raises(ValueError):
            frame_ids(spec, n, "a")


def _host_only(cls):
    """An instance with no model behind it: run()'s checks raise before anything reaches the device."""
    obj = cls.__new__(cls)
    obj.device = "cpu"
    return obj


def test_run_input_validation():
    tt = _host_only(TrackedTePose)
    f = torch.zeros(3, 2048)
    bad = [
        {"a": (0, torch.zeros(3, 2047))},                    # feature width
        {"a": (0, torch.zeros(0, 2048))},                    # no frames
        {"a": (0, torch.zeros(2048))},                       # not [n,2048]
        {"a": ([0, 1], f)},                                  # frame ids of the wrong length
        {"a": ([0, 2, 1], f)},                               # not increasing
        {"a": (-1, f)},                                      # negative first frame
    ]
    for case in bad:
        with pytest.raises(ValueError):
            tt.run(case)
    with pytest.raises(ValueError, match="unknown tracks"):
        tt.run({"a": (0, f)}, theta_input={"b": torch.zeros(3, 85)})

    tv = _host_only(TrackedVideoTePose)
    frames = torch.zeros(4, 8, 8, 3, dtype=torch.uint8)
    boxes = np.zeros((3, 5))
    for fr, tracks in ((frames.float(), {"a": ([0, 1, 2], boxes)}),
                       (frames[0], {"a": ([0, 1, 2], boxes)}),
                       (frames, {"a": ([0, 1, 2], np.zeros((3, 6)))}),   # boxes carry no frame field
                       (frames, {"a": ([0, 1], boxes)}),
                       (frames, {"a": ([1, 2, 4], boxes)}),              # frame 4 of a 4-frame clip
                       (frames, {"a": ([2, 1, 3], boxes)})):
        with pytest.raises(ValueError):
            tv.run(fr, tracks)
    with pytest.raises(ValueError, match="unknown tracks"):
        tv.run(frames, {"a": ([0, 1, 2], boxes)}, theta_input={"b": torch.zeros(3, 85)})


# ------------------------------------------------------------------------------------------------ GPU: the kernels
def _bits(t):
    return t.contiguous().view(torch.int32)


def _ref_push(x, feats, src, op, S, T):
    y = x.clone()
    for s in range(S):
        o, r = int(op[s]), int(src[s])
        if o not in (1, 2) or not 0 <= r < S:
            continue
        if o == 2:
            y[s, :, :COLS] = 0
        else:
            y[s, :T - 1, :2048] = x[s, 1:, :2048]
        y[s, T - 1, :2048] = feats[r]
    return y


def _ref_commit(x, theta, op, S, T):
    y = x.clone()
    for s in range(S):
        if int(op[s]) in (1, 2):
            y[s, :T - 2, 2048:COLS] = x[s, 1:T - 1, 2048:COLS]
            y[s, T - 2, 2048:COLS] = theta[s]
    return y


def _buffers(S, T, ld, g):
    """x [S+1,T,ld] NaN outside the S rows and in the ld padding; feats [S+2,2048] and theta [S+1,85] NaN beyond S rows."""
    x = torch.full((S + 1, T, ld), float("nan"))
    x[:S, :, :COLS] = torch.randn(S, T, COLS, generator=g)
    feats = torch.full((S + 2, 2048), float("nan"))
    feats[:S] = torch.randn(S, 2048, generator=g)
    theta = torch.full((S + 1, 85), float("nan"))
    theta[:S] = torch.randn(S, 85, generator=g)
    return x, feats, theta


def _launch(x, S, T, ld, feats, theta, tab):
    from tepose_b200 import _native as nv
    L = nv.lib()
    nv.check(L.tp_window_slots_push(nv.ptr(x), S, T, ld, nv.ptr(feats), nv.ptr(tab[1]), nv.ptr(tab[0]), nv.stream()))
    nv.check(L.tp_window_slots_commit(nv.ptr(x), S, T, ld, nv.ptr(theta), nv.ptr(tab[0]), nv.stream()))


@pytest.mark.gpu
@pytest.mark.parametrize("ld", [COLS, COLS + 7])
@pytest.mark.parametrize("T", [2, 4, 16])
@pytest.mark.parametrize("S", [1, 5, 32])
def test_slot_kernels_bit_exact(S, T, ld):
    from tepose_b200 import _native as nv
    g = torch.Generator().manual_seed(S * 100 + T + ld)
    x, feats, theta = _buffers(S, T, ld, g)
    op = torch.randint(0, 3, (S,), generator=g, dtype=torch.int32)
    if S >= 3:
        op[:3] = torch.tensor([0, 1, 2], dtype=torch.int32)          # every op on mixed rows
    src = torch.randperm(S, generator=g).to(torch.int32)
    tab = torch.stack([op, src]).to(DEV)
    xd, fd, td = x.to(DEV), feats.to(DEV), theta.to(DEV)
    L = nv.lib()
    nv.check(L.tp_window_slots_push(nv.ptr(xd), S, T, ld, nv.ptr(fd), nv.ptr(tab[1]), nv.ptr(tab[0]), nv.stream()))
    torch.cuda.synchronize()
    want = _ref_push(x, feats, src, op, S, T)
    assert torch.equal(_bits(xd.cpu()), _bits(want))
    nv.check(L.tp_window_slots_commit(nv.ptr(xd), S, T, ld, nv.ptr(td), nv.ptr(tab[0]), nv.stream()))
    torch.cuda.synchronize()
    want = _ref_commit(want, theta, op, S, T)
    assert torch.equal(_bits(xd.cpu()), _bits(want))
    assert torch.equal(_bits(fd.cpu()), _bits(feats)) and torch.equal(_bits(td.cpu()), _bits(theta))


@pytest.mark.gpu
def test_slot_kernels_reject_invalid_arguments():
    from tepose_b200 import _native as nv
    L = nv.lib()
    S, T, ld = 3, 4, COLS
    g = torch.Generator().manual_seed(5)
    x, feats, theta = (t.to(DEV) for t in _buffers(S, T, ld, g))
    tab = torch.tensor([[1, 2, 0], [0, 1, 2]], dtype=torch.int32, device=DEV)
    keep = x.clone()
    xp, fp, tp_, op, sp, st = nv.ptr(x), nv.ptr(feats), nv.ptr(theta), nv.ptr(tab[0]), nv.ptr(tab[1]), nv.stream()
    off = ctypes.c_void_p(x.data_ptr() + 2)
    push = {"null x": (None, S, T, ld, fp, sp, op), "null feats": (xp, S, T, ld, None, sp, op),
            "null src": (xp, S, T, ld, fp, None, op), "null op": (xp, S, T, ld, fp, sp, None),
            "S = 0": (xp, 0, T, ld, fp, sp, op), "S < 0": (xp, -2, T, ld, fp, sp, op), "T = 1": (xp, S, 1, ld, fp, sp, op),
            "ld = 2132": (xp, S, T, ld - 1, fp, sp, op), "x 2 bytes off": (off, S, T, ld, fp, sp, op)}
    for name, a in push.items():
        assert L.tp_window_slots_push(*a, st) == -1, name
    commit = {"null x": (None, S, T, ld, tp_, op), "null theta": (xp, S, T, ld, None, op), "null op": (xp, S, T, ld, tp_, None),
              "S = 0": (xp, 0, T, ld, tp_, op), "T = 1": (xp, S, 1, ld, tp_, op), "ld = 2132": (xp, S, T, ld - 1, tp_, op),
              "x 2 bytes off": (off, S, T, ld, tp_, op)}
    for name, a in commit.items():
        assert L.tp_window_slots_commit(*a, st) == -1, name
    torch.cuda.synchronize()
    assert torch.equal(_bits(x), _bits(keep))                        # nothing was launched


@pytest.mark.gpu
def test_captured_slot_kernels_follow_the_table():
    """One captured push + commit, replayed with rewritten tables; out-of-range ops and src leave their rows untouched."""
    S, T, ld = 5, 4, COLS + 3
    g = torch.Generator().manual_seed(9)
    x, feats, theta = _buffers(S, T, ld, g)
    xd, fd, td = x.to(DEV), feats.to(DEV), theta.to(DEV)
    tab = torch.tensor([[2, 2, 2, 2, 2], [0, 1, 2, 3, 4]], dtype=torch.int32, device=DEV)
    _launch(xd, S, T, ld, fd, td, tab)                               # eager once
    torch.cuda.synchronize()
    want = _ref_commit(_ref_push(x, feats, tab[1].cpu(), tab[0].cpu(), S, T), theta, tab[0].cpu(), S, T)
    assert torch.equal(_bits(xd.cpu()), _bits(want))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        _launch(xd, S, T, ld, fd, td, tab)
    tables = [([1, 0, 1, 2, 1], [4, 0, 3, 1, 2]),
              ([3, -1, 1, 1, 2], [0, 0, S, -1, S + 7]),                 # bad op, bad op, src = S, src < 0, src far out
              ([0, 1, 0, 1, 1], [0, 2, 0, 4, 3])]
    for op, src in tables:
        tab.copy_(torch.tensor([op, src], dtype=torch.int32))
        new_f = torch.randn(S, 2048, generator=g)
        new_t = torch.randn(S, 85, generator=g)
        fd[:S].copy_(new_f)
        td[:S].copy_(new_t)
        feats[:S], theta[:S] = new_f, new_t
        graph.replay()
        torch.cuda.synchronize()
        # the commit of a slot with a bad src still rolls its ring when its op is 1 or 2, as the kernel contract says
        want = _ref_commit(_ref_push(want, feats, torch.tensor(src), torch.tensor(op), S, T), theta, torch.tensor(op), S, T)
        assert torch.equal(_bits(xd.cpu()), _bits(want)), (op, src)


# ------------------------------------------------------------------------------------------------ GPU: per-track equality
@pytest.fixture(scope="module")
def stream_models():
    """TePose T4 L1 H64 and VIBE L2 H32 (the configuration of the windowed-loop golden), fp32."""
    from oracle import torch_ref
    from tepose_b200.synthetic import build_synthetic_model, build_synthetic_vibe
    model, _ = build_synthetic_model(SEED, 4, 1, 64, "fp32", DEV)
    vibe, _ = build_synthetic_vibe(SEED, 4, 2, 32, True, False, True, "fp32", DEV)
    return model, vibe, torch_ref.SmplModel.synthetic(SEED).J_regressor_h36m


# 15 frames, T = 4, 4 slots.  C ends at frame 5 and D (seeded) takes its slot; E is missed at frames 4 and 5 and ends at 10, when
# G (exactly T frames) takes its slot; F is shorter than T; B starts mid-clip in the slot F left.
CLIP = {"A": np.arange(0, 15), "C": np.arange(0, 6), "E": np.array([1, 2, 3, 6, 7, 8, 9, 10]), "F": np.arange(2, 5),
        "B": np.arange(5, 15), "D": np.arange(7, 15), "G": np.arange(11, 15)}
SLOTS = {"A": 0, "C": 1, "E": 2, "F": 3, "B": 3, "D": 1, "G": 2}
SEEDED = "D"


def _slots(frames, S):
    """The slot each track of a clip gets: the bookkeeping replayed over the clip's schedule."""
    t, slot = SlotTable(S), {}
    for _, present, ending in schedule(frames):
        p = t.plan([i for i, _ in present])
        t.apply(p)
        for i, s in zip(p.ids, p.slots):
            slot.setdefault(i, s)
        for i in ending:
            t.end(i)
    return slot


@pytest.mark.gpu
def test_tracked_run_equals_windowed_run_per_track(stream_models):
    """Track b's outputs are row slot(b) of WindowedTePose(batch=4).run on a batch whose row slot(b) holds b's own frames, in
    order and without gaps: every kernel on the path computes a row from that row's inputs alone at a fixed batch."""
    from tepose_b200.stream import WindowedTePose
    model, vibe, J = stream_models
    S, T = 4, 4
    g = torch.Generator().manual_seed(11)
    feats = {i: torch.randn(len(f), 2048, generator=g) for i, f in CLIP.items()}
    seed = 0.1 * torch.randn(T - 1, 85, generator=g)
    assert _slots(CLIP, S) == SLOTS
    tt = TrackedTePose(model, vibe, J_regressor=J, slots=S)
    got = tt.run({i: (CLIP[i], feats[i]) for i in CLIP}, theta_input={SEEDED: seed})
    assert set(got) == set(CLIP) - {"F"}                     # F has fewer than T frames
    for i in got:
        n, s = len(CLIP[i]), SLOTS[i]
        F = torch.randn(S, n, 2048, generator=g)
        F[s] = feats[i]
        kw = {}
        if i == SEEDED:
            th = 0.1 * torch.randn(S, T - 1, 85, generator=g)
            th[s] = seed
            kw = dict(theta_input=th)
        want = WindowedTePose(model, vibe, J_regressor=J, batch=S).run(F.to(DEV), **kw)
        for k in KEYS:
            assert got[i][k].shape == want[k][s].shape, (i, k)
            assert torch.equal(got[i][k], want[k][s]), (i, k, float((got[i][k] - want[k][s]).abs().max()))
    again = tt.run({i: (CLIP[i], feats[i]) for i in CLIP}, theta_input={SEEDED: seed})      # the same object: no state leaks
    for i in got:
        for k in KEYS:
            assert torch.equal(again[i][k], got[i][k]), (i, k)


@pytest.mark.gpu
def test_tracked_push_without_bootstrap_model_needs_a_seed(stream_models):
    model, _, J = stream_models
    T = 4
    tt = TrackedTePose(model, None, J_regressor=J, slots=2)
    f = torch.randn(1, 2048, device=DEV)
    with pytest.raises(ValueError, match="without theta_input"):
        tt.push(f, ["a"])
    seed = torch.zeros(T - 1, 85)
    outs = [tt.push(f, ["a"], theta_input={"a": seed} if t == 0 else None) for t in range(T + 1)]
    assert all(o == {} for o in outs[:T - 1])
    assert outs[T - 1]["a"]["theta"].shape == (1, 85) and outs[T]["a"]["verts"].shape == (1, 6890, 3)


# ------------------------------------------------------------------------------------------------ GPU: frames -> meshes
def _video_clip(H, W, N, tracks):
    """N frames and {id: (frame ids, boxes [n,5])}: people walking in from the sides, leaving and coming back."""
    from oracle import crop_ref
    frames = torch.from_numpy(crop_ref.sample_frames(SEED + H, N, H, W))
    out = {}
    for j, (i, f) in enumerate(tracks.items()):
        b = np.array([(W * (0.15 + 0.2 * j) + 1.7 * t, H * (0.5 - 0.05 * j) - 0.9 * t, W * 0.25 + t, H * 0.6 - t, 1.2)
                      for t in f])
        out[i] = (f, b)
    return frames, out


def _features_of(hmr, frames, tracks, S):
    """Per-track features as TrackedVideoTePose computes them: per frame, the present people's crops compacted and padded to
    bucket(n, S) rows, through HMR.features_from_frames."""
    frames_by = {i: f for i, (f, _) in tracks.items()}
    rows = {i: [] for i in tracks}
    fr = frames.to(DEV)
    with torch.no_grad():
        for f, present, _ in schedule(frames_by):
            crops = np.array([(0,) + tuple(tracks[i][1][k]) for i, k in present])
            feats = hmr.features_from_frames(fr[f:f + 1], compact_crops(crops, bucket(len(present), S)))
            for j, (i, _) in enumerate(present):
                rows[i].append(feats[j])
    return {i: (frames_by[i], torch.stack(rows[i])) for i in tracks}


VIDEO_TRACKS = {"p": np.arange(0, 9), "q": np.array([2, 3, 4, 7, 8]), "r": np.arange(1, 4), "s": np.arange(4, 9)}


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,precision", [(97, 131, "bf16"), (97, 131, "fp32_tc"), (1080, 1920, "bf16")])
def test_tracked_video_run_equals_tracked_run_on_hmr_features(stream_models, H, W, precision):
    from tepose_b200.synthetic import build_synthetic_hmr
    model, vibe, J = stream_models
    S = 4
    hmr = build_synthetic_hmr(SEED, DEV, precision=precision)
    tracks = VIDEO_TRACKS if H < 1000 else {"p": np.arange(0, 6), "q": np.array([1, 2, 4, 5])}
    N = 1 + max(int(f[-1]) for f in tracks.values())
    frames, tracks = _video_clip(H, W, N, tracks)
    want = TrackedTePose(model, vibe, J_regressor=J, slots=S).run(_features_of(hmr, frames, tracks, S))
    tv = TrackedVideoTePose(hmr, model, vibe, J_regressor=J, slots=S)
    got = tv.run(frames.to(DEV), tracks)
    assert set(got) == set(want) and set(got) == {i for i, (f, _) in tracks.items() if len(f) >= 4}
    for i in want:
        for k in KEYS:
            assert torch.equal(got[i][k], want[i][k]), (i, k, float((got[i][k] - want[i][k]).abs().max()))
    again = tv.run(frames, tracks)                           # a second clip through the same graphs, frames from the host
    for i in want:
        for k in KEYS:
            assert torch.equal(again[i][k], want[i][k]), (i, k)


@pytest.mark.gpu
def test_tracked_video_push_replays_graphs_only(stream_models, monkeypatch):
    """Pushed frame by frame at S = 8 from pinned host frames: a push in which no track reaches its T-th frame launches nothing
    itself once its graphs exist and replays the bucket graph of its occupancy (3 people: the 4-crop graph), then the push and
    step graphs.  More live tracks than slots raises."""
    from tepose_b200 import _native as nv
    from tepose_b200.synthetic import build_synthetic_hmr
    model, vibe, J = stream_models
    S, T = 8, 4
    hmr = build_synthetic_hmr(SEED, DEV)
    frames, tracks = _video_clip(97, 131, 9, VIDEO_TRACKS)
    want = TrackedVideoTePose(hmr, model, vibe, J_regressor=J, slots=S).run(frames.to(DEV), tracks)

    tv = TrackedVideoTePose(hmr, model, vibe, J_regressor=J, slots=S)
    replayed = []
    real = torch.cuda.CUDAGraph.replay
    monkeypatch.setattr(torch.cuda.CUDAGraph, "replay", lambda self: (replayed.append(self), real(self))[1])

    def names():
        tr = tv.tracker
        named = {id(tr._push_graph): "push", id(tr._step_graph): "step"}
        named.update({id(b["graph"]): f"bucket{nb}" for nb, b in tv.buckets.items()})
        return [named.get(id(g), "?") for g in replayed]

    pinned = frames.pin_memory()
    frames_by = {i: f for i, (f, _) in tracks.items()}
    got = {i: [] for i in tracks}
    steady_pushes = 0
    for f, present, ending in schedule(frames_by):
        nb = bucket(len(present), S)
        steady = (tv.tracker._push_graph is not None and nb in tv.buckets) and all(k + 1 != T for _, k in present)
        replayed.clear()
        before = nv.lib().tp_launch_count()
        out = tv.push(pinned[f:f + 1], {i: (0,) + tuple(tracks[i][1][k]) for i, k in present})
        launched = nv.lib().tp_launch_count() - before
        assert names() == [f"bucket{nb}", "push", "step"], (f, names())
        if len(present) == 3:
            assert nb == 4
        if steady:
            steady_pushes += 1
            assert launched == 0, (f, launched)
        for i, k in present:
            if i in out:
                got[i].append(out[i]["verts"].clone())
        for i in ending:
            tv.end(i)
    assert steady_pushes >= 3 and any(len(p) == 3 for _, p, _ in schedule(frames_by))
    for i in want:
        assert torch.equal(torch.cat(got[i]), want[i]["verts"]), i
    assert set(tv.buckets) == {bucket(len(p), S) for _, p, _ in schedule(frames_by)}

    small = TrackedVideoTePose(hmr, model, vibe, J_regressor=J, slots=2)
    with pytest.raises(ValueError, match="push 0: 3 live tracks for 2 slots"):
        small.push(pinned[:1], {i: (0, 60.0, 50.0, 30.0, 60.0, 1.2) for i in "abc"})
