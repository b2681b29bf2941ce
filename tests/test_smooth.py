"""Pose smoothing (tepose_b200.smooth, csrc/smooth.cu, the smooth= option of tepose_b200.tracks).  CPU: the kernel's explicit
float32 recurrence against the restated reference filter bit for bit, the per-slot filter table from the slot bookkeeping, and
the smooth= checks.  GPU: tp_one_euro_filter bit for bit against that recurrence, smooth_pose against the reference's per-frame
form, and the per-frame smoothing of TrackedTePose / TrackedVideoTePose against the oracle filter over each track's own rows."""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import smooth_ref
from tepose_b200.smooth import SMOOTH_KEYS, smooth_params
from tepose_b200.tracks import SlotTable, TrackedTePose, bucket, schedule, smooth_table

DEV = "cuda:0"
SEED = 71
KEYS = ("theta", "verts", "kp_2d", "kp_3d", "rotmat")
PARAMS = [(0.004, 0.7), (1.0, 0.0), (0.0, 0.0), (0.004, 50.0)]


def _poses(n, c, seed):
    """[n,c] float32 axis-angle-like rows: a slow random walk with jumps of about +-pi (a rotation crossing the wrap-around)."""
    rng = np.random.default_rng(seed)
    x = np.cumsum(0.05 * rng.standard_normal((n, c)), 0) + rng.uniform(-1, 1, (1, c))
    jumps = rng.random((n, c)) < 0.03
    x += np.cumsum(jumps * rng.choice([-math.pi, math.pi], (n, c)), 0)
    return x.astype(np.float32)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _bits_t(t):
    return t.contiguous().view(torch.int32)


# ------------------------------------------------------------------------------------------------ CPU: arithmetic
@pytest.mark.parametrize("params", PARAMS)
@pytest.mark.parametrize("n", [1, 2, 300])
def test_f32_recurrence_equals_reference_filter(n, params):
    x = _poses(n, 72, n)
    want = smooth_ref.filter_pose(x, *params)
    got, _ = smooth_ref.one_euro_f32(x, *params)
    assert np.array_equal(_bits(got), _bits(want))
    assert np.array_equal(_bits(got[0]), _bits(x[0]))                  # frame 0 passes through


def test_f32_recurrence_continues_from_its_state():
    x = _poses(300, 72, 5)
    whole, st_whole = smooth_ref.one_euro_f32(x, 0.004, 0.7)
    a, st = smooth_ref.one_euro_f32(x[:17], 0.004, 0.7)
    b, st = smooth_ref.one_euro_f32(x[17:18], 0.004, 0.7, st)
    c, st = smooth_ref.one_euro_f32(x[18:], 0.004, 0.7, st)
    assert np.array_equal(_bits(np.concatenate([a, b, c])), _bits(whole))
    assert all(np.array_equal(_bits(u), _bits(v)) for u, v in zip(st, st_whole))


# ------------------------------------------------------------------------------------------------ CPU: the per-slot table
def test_smooth_table_from_the_slot_bookkeeping():
    """T = 3, 2 slots.  a: start, output from its 3rd push, missed once (count 0, state kept), then one row per push.  b: ends,
    c takes its slot and starts its filter at its own 3rd push.  With a bootstrap model the 3rd push filters eagerly."""
    T, S = 3, 2
    pushes = [["a", "b"], ["a", "b"], ["a", "b"], ["b"], ["a"], ["a", "c"], ["a", "c"], ["c", "a"]]
    ends = {3: ["b"]}
    want = {  # push -> (count, reset, boot) without a bootstrap model, then with one
        0: (([0, 0], [0, 0], []), ([0, 0], [0, 0], [])),
        2: (([1, 1], [1, 1], []), ([0, 0], [0, 0], [0, 1])),
        3: (([0, 1], [0, 0], []), ([0, 1], [0, 0], [])),          # a missed: count 0
        4: (([1, 0], [0, 0], []), ([1, 0], [0, 0], [])),          # a continues from its state
        5: (([1, 0], [0, 0], []), ([1, 0], [0, 0], [])),          # c took b's slot: nothing before its 3rd frame
        7: (([1, 1], [0, 1], []), ([1, 0], [0, 0], [1])),         # c's 3rd frame: reset (or bootstrap) in slot 1
    }
    for boot_model in (False, True):
        t = SlotTable(S)
        for k, ids in enumerate(pushes):
            p = t.plan(ids)
            got = smooth_table(p, S, T, boot_model)
            if k in want:
                assert got == want[k][boot_model], (k, boot_model, got)
            t.apply(p)
            for i in ends.get(k, []):
                t.end(i)


def test_smooth_argument_is_checked():
    assert smooth_params(None) is None
    assert smooth_params((0.004, 0.7)) == (0.004, 0.7) and smooth_params([1, 0]) == (1.0, 0.0)
    for bad in [(0.004,), (0.004, 0.7, 1.0), (-0.1, 0.7), (0.004, -1.0), (float("nan"), 0.7), (0.004, float("inf")),
                ("0.004", 0.7), (True, 0.7), 0.7, "ab"]:
        with pytest.raises(ValueError):
            smooth_params(bad)
        with pytest.raises(ValueError):                                # checked before the model is touched
            TrackedTePose(None, smooth=bad)


# ------------------------------------------------------------------------------------------------ GPU: the kernel
def _filter(x, out, state, count, reset, S, K, C, mc, beta, ldx=None, ldo=None):
    from tepose_b200 import _native as nv
    ldx = ldx or (x.stride(0), x.stride(1))
    ldo = ldo or (out.stride(0), out.stride(1))
    return nv.lib().tp_one_euro_filter(ctypes.c_void_p(x.data_ptr()), ldx[0], ldx[1], ctypes.c_void_p(out.data_ptr()), ldo[0],
                                       ldo[1], ctypes.c_void_p(state.data_ptr()), ctypes.c_void_p(count.data_ptr()),
                                       ctypes.c_void_p(reset.data_ptr()), S, K, C, mc, beta, nv.stream())


def _case(S, K, seed):
    """x [S,K,85] (the 72 channels in columns 3..74, row stride 85), counts from 1 to K with some 0 and two out of range, mixed
    resets and random starting states."""
    rng = np.random.default_rng(seed)
    x = np.full((S, K, 85), np.nan, np.float32)
    for s in range(S):
        x[s, :, 3:75] = _poses(K, 72, seed * 100 + s)
    count = rng.integers(1, K + 1, S)
    count[rng.random(S) < 0.2] = 0
    if S > 1:
        count[0], count[-1] = K, 1
    if S > 4:
        count[2], count[3] = -3, K + 5                                # outside [0, K]: treated as 0
    reset = (rng.random(S) < 0.5).astype(np.int32)
    state = np.stack([_poses(2, 72, seed + 7)[0][None].repeat(S, 0) + rng.standard_normal((S, 72)).astype(np.float32),
                      0.1 * rng.standard_normal((S, 72)).astype(np.float32)], 1).astype(np.float32)
    return x, count.astype(np.int32), reset, state


def _want(x, count, reset, state, K, mc, beta):
    S = x.shape[0]
    out = np.full((S, K, 72), np.nan, np.float32)
    st = state.copy()
    for s in range(S):
        n = int(count[s])
        if not 0 < n <= K:
            continue
        o, (xp, dxp) = smooth_ref.one_euro_f32(x[s, :n, 3:75], mc, beta, None if reset[s] else (state[s, 0], state[s, 1]))
        out[s, :n], st[s, 0], st[s, 1] = o, xp, dxp
    return out, st


@pytest.mark.gpu
@pytest.mark.parametrize("params", [(0.004, 0.7), (0.0, 0.0), (0.004, 50.0)])
@pytest.mark.parametrize("S", [1, 5, 33])
def test_filter_kernel_bit_exact(S, params):
    K = 1000
    x, count, reset, state = _case(S, K, S)
    if S == 1:
        count[0] = K
    want, want_state = _want(x, count, reset, state, K, *params)
    xd = torch.from_numpy(x).to(DEV)
    out = torch.full((S, K, 72), float("nan"), device=DEV)
    st = torch.from_numpy(state).to(DEV)
    cd, rd = torch.from_numpy(count).to(DEV), torch.from_numpy(reset).to(DEV)
    view = xd[:, :, 3:75]
    assert _filter(view, out, st, cd, rd, S, K, 72, *params) == 0
    torch.cuda.synchronize()
    assert np.array_equal(_bits(out.cpu().numpy()), _bits(want))        # rows beyond count stay NaN: nothing written
    assert np.array_equal(_bits(st.cpu().numpy()), _bits(want_state))
    assert np.array_equal(_bits(xd.cpu().numpy()), _bits(x))

    # the same sequences in chunks of several calls, the state carried between them
    out2 = torch.full((S, K, 72), float("nan"), device=DEV)
    st2 = torch.from_numpy(state).to(DEV)
    zero = torch.zeros(S, dtype=torch.int32, device=DEV)
    lo = 0
    for j, c in enumerate([1, 7, 64, 300, 1000]):
        c = min(c, K - lo)
        if c <= 0:
            break
        n = np.where((count >= 0) & (count <= K), np.clip(count - lo, 0, c), 0).astype(np.int32)
        assert _filter(view[:, lo:], out2[:, lo:], st2, torch.from_numpy(n).to(DEV), rd if j == 0 else zero, S, c, 72,
                       *params) == 0
        lo += c
    torch.cuda.synchronize()
    assert np.array_equal(_bits(out2.cpu().numpy()), _bits(want))
    assert np.array_equal(_bits(st2.cpu().numpy()), _bits(want_state))


@pytest.mark.gpu
def test_filter_kernel_rejects_invalid_arguments():
    from tepose_b200 import _native as nv
    S, K, C = 3, 4, 72
    x = torch.randn(S, K, 85, device=DEV)
    out = torch.full((S, K, C), float("nan"), device=DEV)
    st = torch.zeros(S, 2, C, device=DEV)
    cnt = torch.full((S,), K, dtype=torch.int32, device=DEV)
    rst = torch.ones(S, dtype=torch.int32, device=DEV)
    L, sp = nv.lib(), nv.stream()
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    xp, op_, sp_, cp, rp = P(x[:, :, 3:]), P(out), P(st), P(cnt), P(rst)
    good = [xp, K * 85, 85, op_, K * C, C, sp_, cp, rp, S, K, C, 0.004, 0.7]
    bad = {"null x": (0, None), "null out": (3, None), "null state": (6, None), "null count": (7, None), "null reset": (8, None),
           "S = 0": (9, 0), "K = 0": (10, 0), "C = 0": (11, 0), "S < 0": (9, -1),
           "x seq stride < C": (1, C - 1), "x row stride < C": (2, C - 1), "out seq stride < C": (4, 0), "out row stride < C": (5, 71),
           "min_cutoff < 0": (12, -0.5), "min_cutoff nan": (12, float("nan")), "min_cutoff inf": (12, float("inf")),
           "beta < 0": (13, -1.0), "beta inf": (13, float("inf"))}
    for name, (k, v) in bad.items():
        a = list(good)
        a[k] = v
        assert L.tp_one_euro_filter(*a, sp) == -1, name
    torch.cuda.synchronize()
    assert bool(torch.isnan(out).all()) and bool((st == 0).all())        # nothing was launched
    assert L.tp_one_euro_filter(*good, sp) == 0
    torch.cuda.synchronize()
    assert not bool(torch.isnan(out).any())


# ------------------------------------------------------------------------------------------------ GPU: smooth_pose
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 75])
def test_smooth_pose_against_reference(n):
    import tepose_b200
    from oracle import synth, torch_ref
    from tests.helpers import base_data_cwd
    seed = 13
    m = torch_ref.SmplModel.synthetic(seed)
    b = synth.make_bodies(seed, n)
    pose = (b["pose_aa"] + 0.3 * _poses(n, 72, n)).astype(np.float32)
    betas = b["betas"].astype(np.float32)
    want_v, want_p, want_j = smooth_ref.smooth_pose(m, pose, betas)
    with base_data_cwd(seed):
        smpl = tepose_b200.SMPL(tepose_b200.SMPL_MODEL_DIR, batch_size=1, create_transl=False).to(DEV)
        default = tepose_b200.smooth_pose(torch.from_numpy(pose).to(DEV), torch.from_numpy(betas).to(DEV))   # builds its own SMPL
    got_v, got_p, got_j = tepose_b200.smooth_pose(torch.from_numpy(pose).to(DEV), torch.from_numpy(betas).to(DEV), smpl=smpl)
    assert got_v.shape == (n, 6890, 3) and got_p.shape == (n, 72) and got_j.shape == (n, 49, 3)
    assert np.array_equal(_bits(got_p.cpu().numpy()), _bits(want_p))
    ev, ej = float(np.abs(got_v.cpu().numpy() - want_v).max()), float(np.abs(got_j.cpu().numpy() - want_j).max())
    assert ev < 1e-4 and ej < 1e-4, (ev, ej)
    for g, d in zip((got_v, got_p, got_j), default):
        assert torch.equal(g, d)
    with pytest.raises(ValueError):
        tepose_b200.smooth_pose(torch.zeros(3, 71, device=DEV), torch.zeros(3, 10, device=DEV), smpl=smpl)
    with pytest.raises(ValueError):
        tepose_b200.smooth_pose(torch.zeros(3, 72, device=DEV), torch.zeros(2, 10, device=DEV), smpl=smpl)


# ------------------------------------------------------------------------------------------------ GPU: per-frame smoothing
@pytest.fixture(scope="module")
def stream_models():
    """TePose T4 L1 H64 and VIBE L2 H32, fp32 (the models of tests/test_tracks.py)."""
    from oracle import torch_ref
    from tepose_b200.synthetic import build_synthetic_model, build_synthetic_vibe
    model, _ = build_synthetic_model(SEED, 4, 1, 64, "fp32", DEV)
    vibe, _ = build_synthetic_vibe(SEED, 4, 2, 32, True, False, True, "fp32", DEV)
    return model, vibe, torch_ref.SmplModel.synthetic(SEED).J_regressor_h36m


# 15 frames, T = 4, 4 slots (the clip of tests/test_tracks.py).  C ends at frame 5 and D (seeded) takes its slot; E is missed at
# frames 4 and 5 and ends at 10, when G (exactly T frames) takes its slot; F is shorter than T; B starts mid-clip in F's slot.
CLIP = {"A": np.arange(0, 15), "C": np.arange(0, 6), "E": np.array([1, 2, 3, 6, 7, 8, 9, 10]), "F": np.arange(2, 5),
        "B": np.arange(5, 15), "D": np.arange(7, 15), "G": np.arange(11, 15)}
SEEDED = "D"


def _check_smoothed(res, smpl, m, params):
    """Every track's smoothed outputs against the oracle filter over its own non-NaN theta rows, SMPL against the oracle and
    against smooth_pose on the same rows."""
    import tepose_b200
    from oracle import torch_ref
    for i, r in res.items():
        rows = ~torch.isnan(r["theta"][:, 0])
        assert bool(rows.any()), i
        assert bool(torch.isnan(r["pose_smooth"][~rows]).all()) and bool(torch.isnan(r["verts_smooth"][~rows]).all())
        th = r["theta"][rows]
        want_p, _ = smooth_ref.one_euro_f32(th[:, 3:75].cpu().numpy(), *params)
        assert np.array_equal(_bits(r["pose_smooth"][rows].cpu().numpy()), _bits(want_p)), i
        want_v, want_j, _ = torch_ref.smpl_forward(m, th[:, 75:].cpu(), pose_aa=torch.from_numpy(want_p))
        ev = float((r["verts_smooth"][rows].cpu() - want_v).abs().max())
        ej = float((r["joints3d_smooth"][rows].cpu() - want_j).abs().max())
        assert ev < 1e-4 and ej < 1e-4, (i, ev, ej)
        v, p, j = tepose_b200.smooth_pose(th[:, 3:75], th[:, 75:], *params, smpl=smpl)
        assert torch.equal(p, r["pose_smooth"][rows]), i
        dv, dj = float((v - r["verts_smooth"][rows]).abs().max()), float((j - r["joints3d_smooth"][rows]).abs().max())
        assert dv < 1e-5 and dj < 1e-5, (i, dv, dj)


@pytest.mark.gpu
@pytest.mark.parametrize("bootstrap", [True, False])
def test_tracked_smoothing_per_track(stream_models, bootstrap):
    from oracle import torch_ref
    model, vibe, J = stream_models
    S, T = 4, 4
    params = (0.004, 0.7)
    g = torch.Generator().manual_seed(11)
    feats = {i: torch.randn(len(f), 2048, generator=g) for i, f in CLIP.items()}
    seeds = {i: 0.1 * torch.randn(T - 1, 85, generator=g) for i in CLIP}
    tin = {SEEDED: seeds[SEEDED]} if bootstrap else seeds
    v = vibe if bootstrap else None
    clip = {i: (CLIP[i], feats[i]) for i in CLIP}
    raw = TrackedTePose(model, v, J_regressor=J, slots=S).run(clip, theta_input=tin)
    tt = TrackedTePose(model, v, J_regressor=J, slots=S, smooth=params)
    got = tt.run(clip, theta_input=tin)
    assert set(got) == set(raw) == set(CLIP) - {"F"}
    for i in got:
        assert set(got[i]) == set(KEYS) | set(SMOOTH_KEYS)
        for k in KEYS:                                                  # NaN rows without a bootstrap model: compare bits
            assert torch.equal(_bits_t(got[i][k]), _bits_t(raw[i][k])), (i, k)
        n = len(CLIP[i])
        assert got[i]["pose_smooth"].shape == (n, 72) and got[i]["joints3d_smooth"].shape == (n, 49, 3)
    _check_smoothed(got, model.regressor.smpl, torch_ref.SmplModel.synthetic(SEED), params)
    again = tt.run(clip, theta_input=tin)                                # the same object: no filter state leaks
    for i in got:
        for k in got[i]:
            assert torch.equal(_bits_t(again[i][k]), _bits_t(got[i][k])), (i, k)


@pytest.mark.gpu
def test_tracked_video_smoothing_push_replays_graphs_only(stream_models):
    """Pushed frame by frame from pinned host frames with smooth on: a steady push launches nothing itself, and the smoothed
    outputs equal those of run()."""
    from tepose_b200 import _native as nv
    from tepose_b200.synthetic import build_synthetic_hmr
    from tepose_b200.tracks import TrackedVideoTePose
    from oracle import crop_ref
    model, vibe, J = stream_models
    S, T, H, W = 8, 4, 97, 131
    hmr = build_synthetic_hmr(SEED, DEV)
    tracks_f = {"p": np.arange(0, 9), "q": np.array([2, 3, 4, 7, 8]), "r": np.arange(1, 4), "s": np.arange(4, 9)}
    frames = torch.from_numpy(crop_ref.sample_frames(SEED + H, 9, H, W))
    tracks = {}
    for j, (i, f) in enumerate(tracks_f.items()):
        tracks[i] = (f, np.array([(W * (0.15 + 0.2 * j) + 1.7 * t, H * (0.5 - 0.05 * j) - 0.9 * t, W * 0.25 + t, H * 0.6 - t, 1.2)
                                  for t in f]))
    want = TrackedVideoTePose(hmr, model, vibe, J_regressor=J, slots=S, smooth=(0.004, 0.7)).run(frames.to(DEV), tracks)
    assert set(want["p"]) == set(KEYS) | set(SMOOTH_KEYS)
    tv = TrackedVideoTePose(hmr, model, vibe, J_regressor=J, slots=S, smooth=(0.004, 0.7))
    pinned = frames.pin_memory()
    got = {i: {k: [] for k in SMOOTH_KEYS} for i in tracks}
    steady_pushes = 0
    for f, present, ending in schedule(tracks_f):
        nb = bucket(len(present), S)
        steady = (tv.tracker._push_graph is not None and nb in tv.buckets) and all(k + 1 != T for _, k in present)
        before = nv.lib().tp_launch_count()
        out = tv.push(pinned[f:f + 1], {i: (0,) + tuple(tracks[i][1][k]) for i, k in present})
        launched = nv.lib().tp_launch_count() - before
        if steady:
            steady_pushes += 1
            assert launched == 0, (f, launched)
        for i in out:
            for k in SMOOTH_KEYS:
                got[i][k].append(out[i][k].clone())
        for i in ending:
            tv.end(i)
    assert steady_pushes >= 3
    for i in want:
        for k in SMOOTH_KEYS:
            assert torch.equal(torch.cat(got[i][k]), want[i][k]), (i, k)
