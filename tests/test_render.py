"""Frame-coordinate cameras and the mesh overlay (tepose_b200.render).  CPU: the fill rule of the contract partitions the pixels,
crop_cam_to_frame / crop_kp_to_frame against the crop transform and the reference formula, the vertex -> face CSR.  GPU:
MeshRenderer.render bit for bit against oracle/render_ref.py on tracked-video meshes, a closed SMPL-sized sphere, overlapping,
off-frame, degenerate and non-finite inputs; composite order, determinism, n = 0, argument checks; render_clip against
per-frame render calls."""
import numpy as np
import pytest
import torch

from oracle import crop_ref, render_ref
from tepose_b200.render import DEFAULT_COLOR, crop_cam_to_frame, crop_kp_to_frame, vertex_faces

DEV = "cuda:0"
SEED = 71


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_fill_rule_partitions_a_triangulated_rectangle(seed):
    """A regular grid of vertices on pixel centres (every sample on an edge or vertex somewhere), random diagonals and windings,
    then the same grid with jittered interior vertices: every pixel strictly inside the rectangle is covered exactly once, no
    pixel twice."""
    rs = np.random.RandomState(seed)
    H, W, gx, gy = 23, 29, 5, 4
    xs = 128 + 256 * np.linspace(2, W - 3, gx + 1).round().astype(np.int64)
    ys = 128 + 256 * np.linspace(2, H - 3, gy + 1).round().astype(np.int64)
    for jitter in (0, 300):
        X, Y = np.meshgrid(xs, ys)
        if jitter:
            X[1:-1, 1:-1] += rs.randint(-jitter, jitter + 1, X[1:-1, 1:-1].shape)
            Y[1:-1, 1:-1] += rs.randint(-jitter, jitter + 1, Y[1:-1, 1:-1].shape)
        tx, ty = [], []
        for j in range(gy):
            for i in range(gx):
                a, b, c, d = (j, i), (j, i + 1), (j + 1, i), (j + 1, i + 1)
                tris = [(a, b, d), (a, d, c)] if rs.rand() < 0.5 else [(a, b, c), (b, d, c)]
                for t in tris:
                    if rs.rand() < 0.5:
                        t = (t[0], t[2], t[1])
                    tx.append([X[v] for v in t])
                    ty.append([Y[v] for v in t])
        tx, ty = np.array(tx), np.array(ty)
        area = (tx[:, 1] - tx[:, 0]) * (ty[:, 2] - ty[:, 0]) - (ty[:, 1] - ty[:, 0]) * (tx[:, 2] - tx[:, 0])
        assert (area != 0).all()
        neg = area < 0
        for a in (tx, ty):
            a[neg, 1], a[neg, 2] = a[neg, 2].copy(), a[neg, 1].copy()
        count = render_ref.coverage(tx, ty, H, W).sum(0)
        assert count.max() == 1
        py, px = np.meshgrid(np.arange(H) * 256 + 128, np.arange(W) * 256 + 128, indexing="ij")
        inside = (px > xs[0]) & (px < xs[-1]) & (py > ys[0]) & (py < ys[-1])
        assert (count[inside] == 1).all()


BOXES = np.array([(300.0, 200.0, 120.0, 120.0, 1.0), (50.5, 420.25, 80.0, 80.0, 1.2),       # square
                  (640.0, 100.0, 60.0, 150.0, 1.1), (-30.0, 700.0, 200.0, 90.0, 0.8)])      # elongated, off-frame
FW, FH = 717, 533


def _cams(n, seed):
    rs = np.random.RandomState(seed)
    return np.stack([rs.uniform(0.5, 1.5, n), rs.uniform(-0.3, 0.3, n), rs.uniform(-0.3, 0.3, n)], 1)


def test_crop_cam_to_frame_maps_through_the_box():
    """A point the crop camera puts at normalised crop coordinates (xn, yn) sits at cx + xn*w*scale/2, cy + yn*h*scale/2 in the
    frame; the frame camera puts it there too (float64)."""
    cam = torch.from_numpy(_cams(len(BOXES), 0))
    oc = crop_cam_to_frame(cam, BOXES, FW, FH).numpy()
    P = np.random.RandomState(1).normal(0, 0.4, (50, 2))
    for i, (cx, cy, w, h, sc) in enumerate(BOXES):
        s, tx, ty = cam[i].numpy()
        xn, yn = s * (P[:, 0] + tx), s * (P[:, 1] + ty)
        want = np.stack([cx + xn * w * sc / 2, cy + yn * h * sc / 2], 1)
        sx, sy, tx2, ty2 = oc[i]
        got = np.stack([(sx * (P[:, 0] + tx2) + 1) * FW / 2, (sy * (P[:, 1] + ty2) + 1) * FH / 2], 1)
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-9)


def test_crop_cam_to_frame_is_the_reference_formula_for_square_boxes():
    """lib/utils/demo_utils.py: convert_crop_cam_to_orig_img with bbox[:, 2] = the crop side w * scale."""
    sq = BOXES[:2]
    cam = _cams(2, 2)
    side = sq[:, 2] * sq[:, 4]
    hw, hh = FW / 2.0, FH / 2.0
    sx = cam[:, 0] * (1.0 / (FW / side))
    sy = cam[:, 0] * (1.0 / (FH / side))
    ref = np.stack([sx, sy, ((sq[:, 0] - hw) / hw / sx) + cam[:, 1], ((sq[:, 1] - hh) / hh / sy) + cam[:, 2]], 1)
    got = crop_cam_to_frame(torch.from_numpy(cam), sq, FW, FH).numpy()
    np.testing.assert_allclose(got, ref, rtol=1e-14, atol=1e-12)


def test_crop_kp_to_frame_inverts_the_crop_transform():
    """Frame points -> patch pixels through the crop's forward affine map (oracle/crop_ref.py) -> normalised crop coordinates
    -> crop_kp_to_frame gives the frame points back (to the float32 rounding of the crop's source points)."""
    rs = np.random.RandomState(3)
    kp, want = [], []
    for cx, cy, w, h, sc in BOXES:
        M = crop_ref.solve_affine(*crop_ref.patch_points(cx, cy, w, h, sc))
        P = np.stack([cx + rs.uniform(-0.6, 0.6, 24) * w * sc, cy + rs.uniform(-0.6, 0.6, 24) * h * sc], 1)
        patch = P @ M[:, :2].T + M[:, 2]
        kp.append(patch / (crop_ref.SIZE / 2) - 1)
        want.append(P)
    got = crop_kp_to_frame(torch.from_numpy(np.stack(kp)), BOXES).numpy()
    np.testing.assert_allclose(got, np.stack(want), rtol=0, atol=2e-3)


def test_vertex_face_csr():
    f = np.array([[0, 1, 2], [2, 1, 3], [3, 3, 0], [4, 0, 2]])
    off, ids = vertex_faces(f, 6)
    assert off.tolist() == [0, 3, 5, 8, 11, 12, 12]
    assert ids.tolist() == [0, 2, 3, 0, 1, 0, 1, 3, 1, 2, 2, 3]          # face 2 repeats vertex 3: listed once per corner
    for v in range(6):
        lst = ids[off[v]:off[v + 1]]
        assert (np.diff(lst) >= 0).all() and sorted(set(lst.tolist())) == sorted(np.nonzero((f == v).any(1))[0].tolist())


# ------------------------------------------------------------------------------------------------ GPU
def _oracle(r, frame, verts, cam, colors):
    return torch.from_numpy(render_ref.render(frame, verts, cam, colors, r.faces, r.vf_offsets, r.vf_faces))


def _check(r, frame, verts, cam, colors=None):
    got = r.render(frame, verts, cam, colors)
    col = torch.tensor(DEFAULT_COLOR).expand(verts.shape[0], 3) if colors is None else colors
    want = _oracle(r, frame, verts, cam, col)
    torch.cuda.synchronize()
    diff = (got.cpu() != want).any(-1)
    assert not diff.any(), f"{int(diff.sum())} pixels differ, first at {diff.nonzero()[0].tolist()}"
    return got


def _frame(H, W, seed):
    return torch.from_numpy(crop_ref.sample_frames(seed, 1, H, W)[0]).to(DEV)


def _people(verts, n, H, W, seed, radius_px):
    """n copies of verts [V,3], each with its own camera: overlapping near the frame centre, the last two partly and fully
    outside the frame when n >= 3; rows [n,V,3], cams [n,4], random colours [n,3]."""
    rs = np.random.RandomState(seed)
    v = np.repeat(verts[None], n, 0).copy()
    v += rs.normal(0, 0.02, v.shape).astype(np.float32)            # each person a slightly different shape
    cams = []
    for i in range(n):
        sx = 2 * radius_px * rs.uniform(0.7, 1.3) / W
        sy = sx * W / H
        cx, cy = rs.uniform(-0.3, 0.3), rs.uniform(-0.3, 0.3)
        if n >= 3 and i == n - 2:
            cx = 0.97                                              # partly outside (right edge)
        if n >= 3 and i == n - 1:
            cy = -3.0                                              # fully outside (above)
        cams.append((sx, sy, cx / sx, cy / sy))
    col = rs.uniform(0.1, 1.0, (n, 3))
    return (torch.tensor(v, dtype=torch.float32, device=DEV), torch.tensor(cams, dtype=torch.float32, device=DEV),
            torch.tensor(col, dtype=torch.float32, device=DEV))


def _mesh(kind):
    if kind == "sphere":
        return render_ref.uv_sphere()
    from tepose_b200.synthetic import make_smpl_model
    m = make_smpl_model(SEED)
    return m["v_template"], m["f"]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,H,W,n,radius", [("sphere", 333, 517, 1, 120), ("sphere", 333, 517, 3, 90),
                                               ("sphere", 333, 517, 8, 70), ("sphere", 1080, 1920, 8, 260),
                                               ("random", 333, 517, 3, 60), ("random", 1080, 1920, 1, 70)])
def test_render_bit_identical_to_oracle(kind, H, W, n, radius):
    from tepose_b200.render import MeshRenderer
    verts, faces = _mesh(kind)
    r = MeshRenderer(faces, H, W)
    frame = _frame(H, W, n + H)
    v, cam, col = _people(verts, n, H, W, n * 7 + W, radius)
    got = _check(r, frame, v, cam, col)
    assert (got != frame).any(-1).float().mean() > 0.001             # something was drawn
    _check(r, frame, v, cam)                                         # default colour


@pytest.mark.gpu
def test_render_degenerate_faces_and_non_finite_vertices():
    """Repeated-vertex faces, a collinear sliver, NaN / inf vertices (one person entirely NaN, as the rows TrackedTePose.run
    returns before a track's first output) and a non-finite camera draw nothing of their own; the rest is bit-identical."""
    from tepose_b200.render import MeshRenderer
    verts, faces = render_ref.uv_sphere()
    faces = faces.copy()
    faces[::97] = np.stack([faces[::97, 0], faces[::97, 0], faces[::97, 1]], 1)
    faces[5::97] = np.stack([faces[5::97, 1], faces[5::97, 2], faces[5::97, 2]], 1)
    faces[7] = (0, 0, 0)
    H, W = 257, 389
    r = MeshRenderer(faces, H, W)
    frame = _frame(H, W, 4)
    v, cam, col = _people(verts, 5, H, W, 9, 80)
    v[0, ::13] = float("nan")
    v[1, 5::17, 2] = float("inf")
    v[2] = float("nan")
    cam[3, 2] = float("nan")
    v[4, :30] = 1e30                                                   # beyond the guard band
    got = _check(r, frame, v, cam, col)
    only_nan = r.render(frame, v[2:4], cam[2:4], col[2:4])
    assert torch.equal(only_nan, frame)


def _quads(z_near, z_far, tilt):
    """Two quads as one mesh: A flat at z_far over x in [-0.5, 0.5]; B at z_near over x in [-0.3, 0.7], tilted so |n_z| = 0.5
    when tilt (shade 0.65 -> 166 for a base of 1), flat otherwise (shade 1 -> 255)."""
    t = np.tan(np.pi / 3) if tilt else 0.0
    A = [(-0.5, -0.5, z_far), (0.5, -0.5, z_far), (0.5, 0.5, z_far), (-0.5, 0.5, z_far)]
    B = [(x, y, z_near + t * (x - 0.2)) for x, y in ((-0.3, -0.4), (0.7, -0.4), (0.7, 0.4), (-0.3, 0.4))]
    return np.array(A + B, np.float32), np.array([[0, 1, 2], [0, 2, 3], [4, 5, 6], [4, 6, 7]])


@pytest.mark.gpu
def test_composite_order_later_person_then_depth():
    from tepose_b200.render import MeshRenderer
    H, W = 64, 96
    frame = torch.zeros(H, W, 3, dtype=torch.uint8, device=DEV)
    cam = torch.tensor([[0.5, 0.5 * W / H, 0.0, 0.0]], device=DEV)
    white = torch.ones(1, 3, device=DEV)
    ov = (W // 2 + 4, H // 2)                                          # a pixel inside both quads
    onlyA = (int(W / 2 - 0.45 * 0.5 * W / 2), H // 2)
    # one person: the nearer quad wins where they overlap, whichever it is in face order
    for near_is_b in (True, False):
        v, f = _quads(-2.0 if near_is_b else 2.0, 0.0, tilt=True)
        r = MeshRenderer(f, H, W, num_verts=8)
        img = _check(r, frame, torch.from_numpy(v).to(DEV)[None], cam, white).cpu()
        assert img[ov[1], ov[0]].tolist() == ([166] * 3 if near_is_b else [255] * 3)
        assert img[onlyA[1], onlyA[0]].tolist() == [255] * 3
    # two people: the later one wins even when it is farther
    v, f = _quads(0.0, 0.0, tilt=False)
    r = MeshRenderer(f[:2], H, W, num_verts=8)
    two = torch.from_numpy(np.stack([v, v + np.float32([0.3, 0.0, 10.0])])).to(DEV)
    cols = torch.tensor([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]], device=DEV)
    img = _check(r, frame, two, cam.expand(2, 4).contiguous(), cols).cpu()
    assert img[ov[1], ov[0]].tolist() == [0, 255, 0]
    assert img[onlyA[1], onlyA[0]].tolist() == [255, 0, 0]
    img = _check(r, frame, two.flip(0).contiguous(), cam.expand(2, 4).contiguous(), cols.flip(0).contiguous()).cpu()
    assert img[ov[1], ov[0]].tolist() == [255, 0, 0]


@pytest.mark.gpu
def test_render_is_deterministic_leaves_the_frame_and_takes_no_people():
    from tepose_b200.render import MeshRenderer
    verts, faces = _mesh("random")
    H, W = 301, 411
    r = MeshRenderer(faces, H, W)
    frame = _frame(H, W, 8)
    keep = frame.clone()
    v, cam, col = _people(verts, 8, H, W, 3, 110)
    a = r.render(frame, v, cam, col)
    b = r.render(frame, v, cam, col)
    assert torch.equal(a, b) and torch.equal(frame, keep)
    empty = r.render(frame, v[:0], cam[:0])
    assert torch.equal(empty, frame) and empty.data_ptr() != frame.data_ptr()
    c = r.render(frame, v, cam, col)                                 # after n = 0 (keys left all-ones, workspace reused)
    assert torch.equal(a, c)


@pytest.mark.gpu
def test_render_rejects_bad_input():
    from tepose_b200 import _native as nv
    from tepose_b200.render import MeshRenderer
    verts, faces = _mesh("sphere")
    for bad in (faces[:, :2], faces.astype(np.float32), np.where(faces == 5, 6890, faces), np.where(faces == 5, -1, faces),
                np.zeros((0, 3), np.int64)):
        with pytest.raises(ValueError):
            MeshRenderer(bad, 32, 32)
    for hw in ((0, 32), (32, 40000)):
        with pytest.raises(ValueError):
            MeshRenderer(faces, *hw)
    H, W = 40, 50
    r = MeshRenderer(faces, H, W)
    frame = _frame(H, W, 1)
    v, cam, col = _people(verts, 2, H, W, 1, 10)
    cases = [(frame.cpu(), v, cam, col), (frame, v.cpu(), cam, col), (frame, v, cam.cpu(), col),
             (frame.float(), v, cam, col), (frame[:, :-1], v, cam, col), (frame[..., :2], v, cam, col),
             (frame, v[:, :-1], cam, col), (frame, v[..., :2], cam, col), (frame, v[0], cam, col),
             (frame, v, cam[:1], col), (frame, v, cam[:, :3], col), (frame, v, cam, col[:1]), (frame, v, cam, col[:, :2])]
    for i, (a, b, c, d) in enumerate(cases):
        with pytest.raises((ValueError, RuntimeError)):
            r.render(a, b, c, d)
    # the C entry point checks its own arguments and launches nothing
    L = nv.lib()
    out = torch.zeros_like(frame)
    ws = nv.workspace(L.tp_render_workspace_bytes(2, 6890, H, W), DEV)
    P = [nv.ptr(frame), nv.ptr(v), nv.ptr(cam), nv.ptr(col), nv.ptr(r.faces), nv.ptr(r.vf_offsets), nv.ptr(r.vf_faces)]
    good = P + [2, 6890, r.F, H, W, nv.ptr(out), nv.ptr(ws), ws.numel(), nv.stream()]
    assert L.tp_render_meshes(*good) == 0
    torch.cuda.synchronize()
    out.zero_()
    for k, val in ((0, None), (1, None), (7, -1), (7, 65536), (9, 0), (9, 65537), (10, 0), (11, 40000), (14, ws.numel() - 1)):
        a = list(good)
        a[k] = val
        assert L.tp_render_meshes(*a) == -1, (k, val)
    assert L.tp_render_workspace_bytes(-1, 6890, H, W) == 0 and L.tp_render_workspace_bytes(1, 6890, 0, W) == 0
    torch.cuda.synchronize()
    assert not out.any()


# ------------------------------------------------------------------------------------------------ GPU: tracked video
@pytest.mark.gpu
def test_render_clip_of_a_tracked_video_run():
    """TrackedVideoTePose.run on a short clip (synthetic SMPL: random faces), then render_clip: every frame equals a render call
    with the tracks present there (in the order of `tracks`, each with crop_cam_to_frame of its own boxes), and every render
    is bit-identical to the oracle."""
    from oracle import torch_ref
    from tepose_b200.render import MeshRenderer, render_clip
    from tepose_b200.synthetic import build_synthetic_hmr, build_synthetic_model, build_synthetic_vibe, make_smpl_model
    from tepose_b200.tracks import TrackedVideoTePose
    model, _ = build_synthetic_model(SEED, 4, 1, 64, "fp32", DEV)
    vibe, _ = build_synthetic_vibe(SEED, 4, 2, 32, True, False, True, "fp32", DEV)
    J = torch_ref.SmplModel.synthetic(SEED).J_regressor_h36m
    hmr = build_synthetic_hmr(SEED, DEV)
    H, W, N = 97, 131, 7
    frames = torch.from_numpy(crop_ref.sample_frames(SEED + H, N, H, W))
    ids = {"p": np.arange(0, 7), "q": np.array([1, 2, 4, 5, 6]), "r": np.arange(2, 4)}
    tracks = {i: (f, np.array([(W * (0.3 + 0.2 * j) + 1.5 * t, H * 0.5 - t, W * 0.3, H * 0.6, 1.2) for t in f]))
              for j, (i, f) in enumerate(ids.items())}
    res = TrackedVideoTePose(hmr, model, vibe, J_regressor=J, slots=4).run(frames.to(DEV), tracks)
    assert set(res) == {"p", "q"}
    r = MeshRenderer(make_smpl_model(SEED)["f"], H, W)
    colors = {"p": (0.9, 0.6, 0.3), "q": (0.3, 0.7, 1.0)}
    clip = render_clip(r, frames, tracks, res, colors)
    drawn = 0
    for fr in range(N):
        present = [(i, int(np.nonzero(ids[i] == fr)[0][0])) for i in tracks if i in res and fr in ids[i]]
        if not present:
            assert torch.equal(clip[fr].cpu(), frames[fr])
            continue
        verts = torch.stack([res[i]["verts"][k] for i, k in present])
        cam = torch.cat([crop_cam_to_frame(res[i]["theta"][k:k + 1, :3], tracks[i][1][k:k + 1], W, H) for i, k in present])
        col = torch.tensor([colors[i] for i, _ in present], device=DEV)
        one = _check(r, frames[fr].to(DEV), verts, cam, col)
        assert torch.equal(clip[fr], one), fr
        drawn += int((one.cpu() != frames[fr]).any(-1).sum())
    assert drawn > 0
