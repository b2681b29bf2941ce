"""GPU: the on-device video front end.  tp_crop_normalize_bf16 against the NumPy restatement of the reference's cv2 crop
(oracle/crop_ref.py, itself pinned against cv2 in tests/test_crop_ref.py), HMR.features_from_frames against
HMR.feature_extractor on the restated crops, and VideoTePose against WindowedTePose on the features HMR extracts."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import crop_ref, torch_ref

DEV = "cuda:0"
SEED = 71
SIZES = [(97, 131), (1080, 1920)]
KEYS = ("theta", "verts", "kp_2d", "kp_3d", "rotmat")


def _bits(t):
    return t.contiguous().view(torch.int16)


@pytest.fixture(scope="module")
def hmr_model():
    from tepose_b200.synthetic import build_synthetic_hmr
    return build_synthetic_hmr(SEED, DEV)


@pytest.fixture(scope="module")
def stream_models():
    """TePose T4 L1 H64 and VIBE L2 H32 (the configuration of the windowed-loop golden), fp32."""
    from tepose_b200.synthetic import build_synthetic_model, build_synthetic_vibe
    model, _ = build_synthetic_model(SEED, 4, 1, 64, "fp32", DEV)
    vibe, _ = build_synthetic_vibe(SEED, 4, 2, 32, True, False, True, "fp32", DEV)
    return model, vibe, torch_ref.SmplModel.synthetic(SEED).J_regressor_h36m


def _crop(frames, table, N, out):
    from tepose_b200 import _native as nv
    F, H, W, _ = frames.shape
    return nv.lib().tp_crop_normalize_bf16(nv.ptr(frames), F, H, W, nv.ptr(table), N, nv.ptr(out), nv.stream())


def _table(rows):
    from tepose_b200.hmr import make_crop_table
    return make_crop_table(np.array(rows, np.float64), DEV)


# ------------------------------------------------------------------------------------------------ the kernel
@pytest.mark.gpu
@pytest.mark.parametrize("H,W", SIZES)
@pytest.mark.parametrize("N", [1, 3, 32])
def test_crop_kernel_is_bit_exact(H, W, N):
    """Output buffer NaN-filled and 2 crops longer than N: every element of the N crops is written, nothing after them."""
    from tepose_b200 import _native as nv
    frames = crop_ref.sample_frames(SEED + H, 2, H, W)
    rows = crop_ref.sample_boxes(SEED, 2, H, W)
    rows = rows[:N] if N != 1 else [rows[1]]
    out = torch.full((N + 2, 224, 224, 4), float("nan"), dtype=torch.bfloat16, device=DEV)
    nv.check(_crop(torch.from_numpy(frames).to(DEV), _table(rows), N, out), "tp_crop_normalize_bf16")
    torch.cuda.synchronize()
    want = crop_ref.crops_nhwc4_bf16(frames, rows)
    got = out[:N].cpu()
    for i in range(N):
        diff = int((_bits(got[i]) != _bits(want[i])).sum())
        assert diff == 0, (i, rows[i], diff)
    assert bool(torch.isnan(out[N:].float()).all())


@pytest.mark.gpu
def test_crop_kernel_rejects_invalid_arguments():
    from tepose_b200 import _native as nv
    L = nv.lib()
    frames = torch.zeros(2, 20, 30, 3, dtype=torch.uint8, device=DEV)
    table = _table([(1, 10.0, 10.0, 8.0, 8.0, 1.2), (0, 5.0, 5.0, 8.0, 8.0, 1.0)])
    bad_frame = _table([(0, 10.0, 10.0, 8.0, 8.0, 1.2), (2, 5.0, 5.0, 8.0, 8.0, 1.0)])
    negative_frame = _table([(-1, 10.0, 10.0, 8.0, 8.0, 1.2)])
    out = torch.full((3, 224, 224, 4), float("nan"), dtype=torch.bfloat16, device=DEV)
    f, t, o, st = nv.ptr(frames), nv.ptr(table), nv.ptr(out), nv.stream()
    raw = ctypes.c_void_p
    cases = {
        "null frames": (None, 2, 20, 30, t, 2, o),
        "null crops": (f, 2, 20, 30, None, 2, o),
        "null out": (f, 2, 20, 30, t, 2, None),
        "N = 0": (f, 2, 20, 30, t, 0, o),
        "N < 0": (f, 2, 20, 30, t, -1, o),
        "F = 0": (f, 0, 20, 30, t, 2, o),
        "H = 0": (f, 2, 0, 30, t, 2, o),
        "W < 0": (f, 2, 20, -30, t, 2, o),
        "out 8 bytes off alignment": (f, 2, 20, 30, t, 2, raw(out.data_ptr() + 8)),
        "crops 2 bytes off alignment": (f, 2, 20, 30, raw(table.data_ptr() + 2), 2, o),
        "frame index == F": (f, 2, 20, 30, nv.ptr(bad_frame), 2, o),
        "frame index < 0": (f, 2, 20, 30, nv.ptr(negative_frame), 1, o),
        "frame index >= F (F = 1)": (f, 1, 20, 30, t, 2, o),
    }
    for name, (fp, F, H, W, tp, N, op) in cases.items():
        assert L.tp_crop_normalize_bf16(fp, F, H, W, tp, N, op, st) == -1, name          # TP_ERR_INVALID
    torch.cuda.synchronize()
    assert bool(torch.isnan(out.float()).all())                                         # nothing was launched
    assert L.tp_crop_normalize_bf16(f, 2, 20, 30, t, 2, o, st) == 0


@pytest.mark.gpu
def test_captured_crop_reads_the_table_at_replay():
    """A captured launch follows boxes rewritten between replays; a frame index gone bad after capture gives zeros."""
    from tepose_b200 import _native as nv
    H, W = 97, 131
    frames = crop_ref.sample_frames(SEED, 2, H, W)
    rows = crop_ref.sample_boxes(SEED + 1, 2, H, W)
    a, b = rows[1:3], rows[5:7]
    fr = torch.from_numpy(frames).to(DEV)
    table = _table(a)
    out = torch.zeros(2, 224, 224, 4, dtype=torch.bfloat16, device=DEV)
    nv.check(_crop(fr, table, 2, out))                      # eager once (checks the frame indices)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        nv.check(_crop(fr, table, 2, out))
    results = []
    for r in (b, a):
        table.copy_(_table(r))
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(_bits(out.cpu()), _bits(crop_ref.crops_nhwc4_bf16(frames, r)))
        results.append(out.clone())
    assert not torch.equal(results[0], results[1])
    table.copy_(_table([(2,) + tuple(a[0][1:]), a[1]]))
    g.replay()
    torch.cuda.synchronize()
    assert bool((_bits(out[0]) == 0).all())
    assert torch.equal(_bits(out[1].cpu()), _bits(crop_ref.crops_nhwc4_bf16(frames, [a[1]])[0]))


# ------------------------------------------------------------------------------------------------ HMR
@pytest.mark.gpu
def test_features_from_frames_equal_feature_extractor_on_the_reference_crops(hmr_model):
    """Same stem input bit for bit (the restated crops rounded to bf16), deterministic GEMMs: identical features."""
    H, W = 1080, 1920
    frames = crop_ref.sample_frames(SEED + 5, 2, H, W)
    rows = crop_ref.sample_boxes(SEED + 5, 2, H, W)[:5]
    with torch.no_grad():
        got = hmr_model.features_from_frames(torch.from_numpy(frames).to(DEV), rows)
        nchw = np.stack([crop_ref.normalize(crop_ref.crop(frames[f], *r)) for f, *r in rows]).transpose(0, 3, 1, 2)
        want = hmr_model.feature_extractor(torch.from_numpy(np.ascontiguousarray(nchw)).to(DEV))
    assert got.shape == (5, 2048)
    assert torch.equal(got, want)


# ------------------------------------------------------------------------------------------------ frames -> meshes
def _clip(B, N, H=180, W=320):
    """N frames [N,H,W,3] and crops [B,N,6] (frame field 0) of B people walking across the frame."""
    frames = crop_ref.sample_frames(SEED + 9, N, H, W)
    crops = np.zeros((B, N, 6))
    for b in range(B):
        for t in range(N):
            crops[b, t] = (0, W * (0.3 + 0.4 * b) + 3.7 * t, H * 0.5 - 1.3 * t, 60 + 2 * t, 120 - t, 1.2)
    return frames, crops


def _features(hmr, frames, crops):
    with torch.no_grad():
        return torch.stack([hmr.features_from_frames(frames[t:t + 1], crops[:, t]) for t in range(frames.shape[0])], 1)


@pytest.mark.gpu
@pytest.mark.parametrize("option", ["default", "bootstrap_frames", "theta_input"])
def test_video_run_equals_windowed_run_on_hmr_features(hmr_model, stream_models, option):
    from tepose_b200 import VideoTePose
    from tepose_b200.stream import WindowedTePose
    model, vibe, J = stream_models
    B, T = 2, 4
    N = T + 5
    frames, crops = _clip(B, N)
    fr = torch.from_numpy(frames).to(DEV)
    kw = {}
    if option == "bootstrap_frames":
        kw = dict(bootstrap_frames=N)
    elif option == "theta_input":
        kw = dict(theta_input=0.1 * torch.randn(T - 1, 85, generator=torch.Generator().manual_seed(3)))
    ws = WindowedTePose(model, vibe, J_regressor=J, batch=B)
    want = ws.run(_features(hmr_model, fr, crops), **kw)
    vt = VideoTePose(hmr_model, model, vibe, J_regressor=J, batch=B)
    got = vt.run(fr, torch.from_numpy(crops).to(DEV), **kw)
    for k in KEYS:
        assert got[k].shape == want[k].shape, k
        assert torch.equal(got[k], want[k]), (k, float((got[k] - want[k]).abs().max()))
    again = vt.run(fr, crops, **kw)                          # a second clip through the same graph
    for k in KEYS:
        assert torch.equal(again[k], want[k]), k


@pytest.mark.gpu
def test_push_frame_by_frame_is_one_graph_replay_per_frame(hmr_model, stream_models):
    """Pinned host frames and host crops, pushed one by one, give what run() gives; once the window is full a push launches
    nothing itself and replays one graph of crop + HMR + window step."""
    from tepose_b200 import VideoTePose, _native as nv
    from tepose_b200.stream import WindowedTePose
    model, vibe, J = stream_models
    B, T = 2, 4
    N = T + 5
    frames, crops = _clip(B, N)
    want = VideoTePose(hmr_model, model, vibe, J_regressor=J, batch=B).run(torch.from_numpy(frames).to(DEV), crops)

    vt = VideoTePose(hmr_model, model, vibe, J_regressor=J, batch=B)
    pinned = torch.from_numpy(frames).pin_memory()
    replays = []
    got = {k: [] for k in KEYS}
    for t in range(N):
        if vt._graph is not None and not replays:
            real = vt._graph.replay
            vt._graph.replay = lambda: (replays.append(1), real())[1]
        before = nv.lib().tp_launch_count()
        out = vt.push(pinned[t:t + 1], crops[:, t])
        launched = nv.lib().tp_launch_count() - before
        if t < T - 1:
            assert out is None
            continue
        if t == T - 1:
            for k in KEYS:
                assert out[k].shape[:2] == (B, T), k
                got[k].append(out[k].clone())
            continue
        if t > T:
            assert launched == 0 and len(replays) == t - T, (t, launched, len(replays))
        for k in KEYS:
            got[k].append(out[k][:, None].clone())
    for k in KEYS:
        assert torch.equal(torch.cat(got[k], 1), want[k]), k

    # launches per replay: the crop, the HMR trunk from NHWC4, and one window step
    x4 = torch.zeros(B, 224, 224, 4, dtype=torch.bfloat16, device=DEV)
    before = nv.lib().tp_launch_count()
    with torch.no_grad():
        hmr_model.features_nhwc4(x4)
    trunk = int(nv.lib().tp_launch_count() - before)
    ws = WindowedTePose(model, vibe, J_regressor=J, batch=B)
    ws.run(_features(hmr_model, torch.from_numpy(frames).to(DEV), crops))
    assert trunk == 75                                       # feature_extractor's 76 without the NCHW -> NHWC conversion
    assert vt.launches_per_replay == 1 + trunk + ws.launches_per_replay, (vt.launches_per_replay, ws.launches_per_replay)
    print(f"launches per push: {vt.launches_per_replay} (window step {ws.launches_per_replay})")
