"""Deterministic synthetic assets for the TePose hot path (benchmarks, tests, smoke runs).

The licensed SMPL model, the SPIN mean parameters and the released checkpoints are
not redistributable and are absent here (SURVEY.md F13), so every test, golden
fixture and bench run uses the SMPL-*shaped* stand-ins below.  Everything is drawn
from ``numpy.random.Generator(PCG64(seed))`` -- never from torch's RNG -- so the
same seed yields the same bytes on any box / torch version and golden fixtures only
need to store the seed, not 93 M weights.

Shapes follow the reference:
  * GRU / Linear parameter shapes and names: /root/reference/lib/models/tepose.py:53-68
    and lib/models/spin.py:215-224 (state_dict keys listed in SURVEY.md App. A.1).
  * init distributions: torch defaults U(+-1/sqrt(H)) for nn.GRU, U(+-1/sqrt(fan_in)) for
    nn.Linear, xavier_uniform(gain=0.01) for dec* (lib/models/spin.py:222-224).
  * SMPL-shaped body model: 6890 vertices, 24 joints, 10 betas, 207 pose-blend rows,
    exactly 4 non-zero skinning weights per vertex (SURVEY.md section 8d recipe).
"""
from __future__ import annotations

import math
import os
import pickle

import numpy as np

NUM_VERTS = 6890
NUM_JOINTS = 24
NUM_BETAS = 10
NUM_POSE_BASIS = 207
INPUT_SIZE = 2133  # 2048 features + 85 theta   (lib/models/tepose.py:54,60)
FEAT_SIZE = 2048
NPOSE = 144

# Kinematic tree of the SMPL body (smplx: parents = kintree_table[0], root = -1).
SMPL_PARENTS = np.array(
    [-1, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19, 20, 21],
    dtype=np.int64,
)

# smplx.vertex_ids['smplh'] picked vertices appended after the 24 posed joints by
# smplx.vertex_joint_selector.VertexJointSelector (face 5, feet 6, hand tips 10).
SMPL_EXTRA_VERTEX_IDS = np.array(
    [332, 6260, 2800, 4071, 583,
     3216, 3226, 3387, 6617, 6624, 6787,
     2746, 2319, 2445, 2556, 2673,
     6191, 5782, 5905, 6016, 6133],
    dtype=np.int64,
)


def _rng(seed: int, stream: int) -> np.random.Generator:
    return np.random.Generator(np.random.PCG64([int(seed), int(stream)]))


def make_smpl_model(seed: int = 0, skinning: str = "random") -> dict:
    """SMPL-shaped random body model (float32 arrays, pkl-style key names).

    skinning="random" (default; what every golden was generated with): each vertex is bound to 4 joints drawn uniformly --
    no locality at all, the worst case for any kernel that shares joint transforms between neighbouring vertices.
    skinning="coherent": the locality of the licensed SMPL asset (consecutive vertex ids belong to the same body part): runs of
    vertices share a primary joint and take the other three from its kinematic neighbourhood (parent, children, grandparent)."""
    g = _rng(seed, 1)
    V, J = NUM_VERTS, NUM_JOINTS
    v_template = (0.3 * g.standard_normal((V, 3))).astype(np.float32)
    shapedirs = (0.01 * g.standard_normal((V, 3, NUM_BETAS))).astype(np.float32)
    posedirs = (0.001 * g.standard_normal((V, 3, NUM_POSE_BASIS))).astype(np.float32)

    J_regressor = np.zeros((J, V), dtype=np.float32)
    for j in range(J):
        idx = g.choice(V, size=16, replace=False)
        w = g.random(16).astype(np.float32) + 0.05
        J_regressor[j, idx] = w / w.sum()

    weights = np.zeros((V, J), dtype=np.float32)
    cols = np.stack([g.permutation(J)[:4] for _ in range(V)])
    if skinning == "coherent":
        par = SMPL_PARENTS
        neigh = []
        for j in range(J):
            cand = [j] + ([int(par[j])] if par[j] >= 0 else []) + [c for c in range(J) if par[c] == j]
            if par[j] >= 0 and par[int(par[j])] >= 0:
                cand.append(int(par[int(par[j])]))
            cand += [c for c in range(J) if c not in cand]            # pad (leaf joints have few neighbours)
            neigh.append(cand[:4])
        run = V // J + 1                                              # ~288 consecutive vertices per body part
        cols = np.stack([np.array(neigh[min(v // run, J - 1)]) for v in range(V)])
    elif skinning != "random":
        raise ValueError(f"skinning must be 'random' or 'coherent', got {skinning!r}")
    w = g.random((V, 4)).astype(np.float32) + 0.05
    w = w / w.sum(axis=1, keepdims=True)
    np.put_along_axis(weights, cols, w, axis=1)

    faces = g.integers(0, V, size=(13776, 3)).astype(np.int64)
    kintree = np.stack([np.where(SMPL_PARENTS < 0, 2 ** 32 - 1, SMPL_PARENTS),
                        np.arange(J)]).astype(np.int64)
    return {
        "v_template": v_template,
        "shapedirs": shapedirs,
        "posedirs": posedirs,
        "J_regressor": J_regressor,
        "weights": weights,
        "kintree_table": kintree,
        "f": faces,
    }


def make_extra_regressors(seed: int = 0, sparse: bool = False) -> dict:
    """J_regressor_extra [9,6890] (lib/models/smpl.py:54,67), J_regressor_h36m [17,6890]
    (evaluate.py:109).  Dense |N(0,1)|/6890 rows per the SURVEY recipe."""
    g = _rng(seed, 2)
    extra = (np.abs(g.standard_normal((9, NUM_VERTS))) / NUM_VERTS).astype(np.float32)
    h36m = (np.abs(g.standard_normal((17, NUM_VERTS))) / NUM_VERTS).astype(np.float32)
    if sparse:
        for m in (extra, h36m):
            keep = g.random(m.shape) < 0.01
            m *= keep
            m /= np.maximum(m.sum(axis=1, keepdims=True), 1e-12)
    return {"J_regressor_extra": extra, "J_regressor_h36m": h36m}


def make_mean_params() -> dict:
    """smpl_mean_params.npz stand-in (keys read at lib/models/spin.py:232-235)."""
    pose = np.tile(np.array([1, 0, 0, 1, 0, 0], dtype=np.float32), NUM_JOINTS)
    shape = np.full((NUM_BETAS,), 0.1, dtype=np.float32)
    cam = np.array([0.9, 0.0, 0.0], dtype=np.float32)
    return {"pose": pose, "shape": shape, "cam": cam}


def write_base_data(dirname: str, seed: int = 0, skinning: str = "random") -> str:
    """Materialise ``data/base_data`` the way lib/core/config.py:31 expects it."""
    os.makedirs(dirname, exist_ok=True)
    with open(os.path.join(dirname, "SMPL_NEUTRAL.pkl"), "wb") as fh:
        pickle.dump(make_smpl_model(seed, skinning), fh)
    ex = make_extra_regressors(seed)
    np.save(os.path.join(dirname, "J_regressor_extra.npy"), ex["J_regressor_extra"])
    np.save(os.path.join(dirname, "J_regressor_h36m.npy"), ex["J_regressor_h36m"])
    np.savez(os.path.join(dirname, "smpl_mean_params.npz"), **make_mean_params())
    return dirname


def _uniform(g, shape, bound):
    return ((g.random(shape, dtype=np.float32) * 2.0 - 1.0) * np.float32(bound)).astype(np.float32)


def make_state_dict(seed: int = 0, n_layers: int = 1, hidden: int = 2048,
                    scale_dec: float = 1.0) -> dict:
    """Encoder + Regressor parameters, keyed exactly like TePose.state_dict()
    (SURVEY.md App. A.1) minus the regressor.smpl.* buffers.  numpy float32."""
    g = _rng(seed, 3)
    H = hidden
    sd = {}
    kH = 1.0 / math.sqrt(H)
    for name, bidir in (("gru_fwd", False), ("gru_rec", True)):
        ndir = 2 if bidir else 1
        for layer in range(n_layers):
            in_sz = INPUT_SIZE if layer == 0 else H * ndir
            for sfx in ([""] if not bidir else ["", "_reverse"]):
                p = f"encoder.{name}."
                sd[p + f"weight_ih_l{layer}{sfx}"] = _uniform(g, (3 * H, in_sz), kH)
                sd[p + f"weight_hh_l{layer}{sfx}"] = _uniform(g, (3 * H, H), kH)
                sd[p + f"bias_ih_l{layer}{sfx}"] = _uniform(g, (3 * H,), kH)
                sd[p + f"bias_hh_l{layer}{sfx}"] = _uniform(g, (3 * H,), kH)

    def linear(prefix, out_f, in_f, xavier_gain=None):
        if xavier_gain is None:
            b = 1.0 / math.sqrt(in_f)
            sd[prefix + ".weight"] = _uniform(g, (out_f, in_f), b)
        else:
            b = xavier_gain * math.sqrt(6.0 / (in_f + out_f))
            sd[prefix + ".weight"] = _uniform(g, (out_f, in_f), b)
        sd[prefix + ".bias"] = _uniform(g, (out_f,), 1.0 / math.sqrt(in_f))

    linear("encoder.linear_fwd", FEAT_SIZE, H)
    linear("encoder.linear_rec", FEAT_SIZE, 2 * H)
    linear("regressor.fc1", 1024, FEAT_SIZE + NPOSE + 13)
    linear("regressor.fc2", 1024, 1024)
    linear("regressor.decpose", NPOSE, 1024, xavier_gain=0.01 * scale_dec)
    linear("regressor.decshape", 10, 1024, xavier_gain=0.01 * scale_dec)
    linear("regressor.deccam", 3, 1024, xavier_gain=0.01 * scale_dec)
    mp = make_mean_params()
    sd["regressor.init_pose"] = mp["pose"][None]
    sd["regressor.init_shape"] = mp["shape"][None]
    sd["regressor.init_cam"] = mp["cam"][None]
    return sd


def make_vibe_state_dict(seed: int = 0, n_layers: int = 2, hidden: int = 1024, add_linear: bool = True,
                         bidirectional: bool = False) -> dict:
    """VIBE.state_dict() layout (lib/models/vibe.py:37-49,82-95) minus regressor.smpl.*: encoder.gru.*,
    encoder.linear.* (when present) and the same regressor.* block as make_state_dict."""
    g = _rng(seed, 6)
    H, D = hidden, (2 if bidirectional else 1)
    kH = 1.0 / math.sqrt(H)
    sd = {}
    for layer in range(n_layers):
        in_sz = FEAT_SIZE if layer == 0 else H * D
        for sfx in ["", "_reverse"][:D]:
            p = "encoder.gru."
            sd[p + f"weight_ih_l{layer}{sfx}"] = _uniform(g, (3 * H, in_sz), kH)
            sd[p + f"weight_hh_l{layer}{sfx}"] = _uniform(g, (3 * H, H), kH)
            sd[p + f"bias_ih_l{layer}{sfx}"] = _uniform(g, (3 * H,), kH)
            sd[p + f"bias_hh_l{layer}{sfx}"] = _uniform(g, (3 * H,), kH)
    if bidirectional or add_linear:
        b = 1.0 / math.sqrt(D * H)
        sd["encoder.linear.weight"] = _uniform(g, (FEAT_SIZE, D * H), b)
        sd["encoder.linear.bias"] = _uniform(g, (FEAT_SIZE,), b)
    sd.update({k: v for k, v in make_state_dict(seed, 1, 32).items() if k.startswith("regressor.")})
    return sd


def make_vibe_input(seed: int, batch: int, seqlen: int) -> np.ndarray:
    """Static features x ~ N(0,1) [B,T,2048] (evaluate.py:233)."""
    return _rng(seed, 7).standard_normal((batch, seqlen, FEAT_SIZE), dtype=np.float32)


def make_input(seed: int, batch: int, seqlen: int) -> np.ndarray:
    """x ~ N(0,1) [B,T,2133] with the newest frame's theta slot zeroed
    (evaluate.py:248-252 leaves input_feat[0,-1,2048:] at zero)."""
    g = _rng(seed, 4)
    x = g.standard_normal((batch, seqlen, INPUT_SIZE), dtype=np.float32)
    x[:, -1, FEAT_SIZE:] = 0.0
    return x


def make_bodies(seed: int, n: int, pose_scale: float = 0.3) -> dict:
    """Config-4 inputs: axis-angle poses, betas and cameras for ``n`` bodies."""
    g = _rng(seed, 5)
    return {
        "pose_aa": (pose_scale * g.standard_normal((n, 72), dtype=np.float32)),
        "pose_6d": g.standard_normal((n, 144), dtype=np.float32),
        "betas": g.standard_normal((n, 10), dtype=np.float32),
        "cam": (np.array([0.9, 0, 0], np.float32) + 0.1 * g.standard_normal((n, 3), dtype=np.float32)),
    }


def make_train_targets(seed: int, n_rows: int) -> dict:
    """Synthetic regression targets for the outputs that carry gradient in TePoseLoss (lib/core/loss.py:93-131):
    kp_2d [n,49,2], the 14 common 3-D joints [n,14,3], theta [n,85]."""
    g = _rng(seed, 901)
    return {"kp_2d": g.standard_normal((n_rows, 49, 2)).astype(np.float32) * 0.5,
            "kp_3d": g.standard_normal((n_rows, 14, 3)).astype(np.float32) * 0.3,
            "theta": g.standard_normal((n_rows, 85)).astype(np.float32) * 0.2}


def synthetic_train_loss(out: dict, tgt: dict):
    """Stand-in for TePoseLoss on the same outputs (its data terms need the licensed datasets): MSE on kp_2d, on
    kp_3d[:, 25:39] (lib/core/loss.py:99) and on theta.  Plain torch ops: the loss is the caller's code, as in the reference."""
    import torch
    t = lambda k: torch.as_tensor(tgt[k], dtype=out[k].dtype, device=out[k].device)
    kp2 = out["kp_2d"].reshape(-1, 49, 2)
    kp3 = out["kp_3d"].reshape(-1, 49, 3)[:, 25:39]
    th = out["theta"].reshape(-1, 85)
    return ((kp2 - t("kp_2d")) ** 2).mean() + ((kp3 - t("kp_3d")) ** 2).mean() * 10.0 + ((th - t("theta")) ** 2).mean()


def build_synthetic_model(seed: int, seqlen: int, n_layers: int, hidden: int, precision: str = "fp32", device="cpu",
                          skinning: str = "random"):
    """tepose_b200.TePose with the synthetic parameters / SMPL-shaped assets of `seed` loaded.
    Returns (model.eval() on `device`, state_dict as numpy)."""
    import contextlib
    import tempfile
    import torch
    from . import TePose

    @contextlib.contextmanager
    def _cwd(path):
        old = os.getcwd()
        os.chdir(path)
        try:
            yield
        finally:
            os.chdir(old)

    with tempfile.TemporaryDirectory() as tmp:
        write_base_data(os.path.join(tmp, "data", "base_data"), seed, skinning)      # asset paths are cwd-relative
        with _cwd(tmp):
            model = TePose(seqlen=seqlen, n_layers=n_layers, hidden_size=hidden, pretrained="", precision=precision)
    sd = make_state_dict(seed, n_layers, hidden)
    own = model.state_dict()
    for k, v in sd.items():
        assert k in own and tuple(own[k].shape) == tuple(v.shape), k
        own[k] = torch.as_tensor(v)
    model.load_state_dict(own, strict=True)
    return model.to(device).eval(), sd


def build_synthetic_vibe(seed: int, seqlen: int, n_layers: int, hidden: int, add_linear: bool = True,
                         bidirectional: bool = False, use_residual: bool = True, precision: str = "fp32", device="cpu"):
    """tepose_b200.vibe.VIBE with the synthetic parameters / SMPL-shaped assets of `seed` loaded.
    Returns (model.eval() on `device`, state_dict as numpy)."""
    import tempfile
    import torch
    from .vibe import VIBE

    old = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        write_base_data(os.path.join(tmp, "data", "base_data"), seed)      # asset paths are cwd-relative
        os.chdir(tmp)
        try:
            model = VIBE(seqlen=seqlen, n_layers=n_layers, hidden_size=hidden, add_linear=add_linear,
                         bidirectional=bidirectional, use_residual=use_residual, pretrained="", precision=precision)
        finally:
            os.chdir(old)
    sd = make_vibe_state_dict(seed, n_layers, hidden, add_linear, bidirectional)
    own = model.state_dict()
    for k, v in sd.items():
        assert k in own and tuple(own[k].shape) == tuple(v.shape), k
        own[k] = torch.as_tensor(v)
    model.load_state_dict(own, strict=True)
    return model.eval().to(device), sd


def make_hmr_state(shapes: dict, seed: int) -> dict:
    """Deterministic synthetic parameters / BatchNorm statistics for an HMR-shaped model (lib/models/spin.py:59-204): `shapes` maps
    state_dict keys to shapes (smpl.* and init_* keys are skipped -- they come from the synthetic base data).  The same function
    fills the unmodified reference model (oracle/make_golden_hmr.py) and tepose_b200.HMR, so the ~25 M weights never have to be stored."""
    out = {}
    for idx, k in enumerate(sorted(shapes)):
        if k.startswith("smpl.") or k.startswith("init_"):
            continue
        shp = tuple(shapes[k])
        rs = np.random.RandomState((seed * 1000003 + idx * 7919) % (2 ** 31 - 1))
        if k.endswith("num_batches_tracked"):
            out[k] = np.zeros(shp, np.int64)
        elif len(shp) == 4:                                   # conv weight: He init, as the reference's constructor draws it
            n = shp[2] * shp[3] * shp[0]
            out[k] = (rs.standard_normal(shp) * np.sqrt(2.0 / n)).astype(np.float32)
        elif len(shp) == 2:                                   # nn.Linear weight
            gain = 0.01 if k.startswith("dec") else 1.0
            out[k] = ((rs.random_sample(shp) * 2 - 1) * gain / np.sqrt(shp[1])).astype(np.float32)
        elif k.endswith("running_var"):
            out[k] = (0.6 + 0.8 * rs.random_sample(shp)).astype(np.float32)
        elif k.endswith("running_mean"):
            out[k] = (0.05 * rs.standard_normal(shp)).astype(np.float32)
        elif k.split(".")[-2].startswith("bn") or k.split(".")[-2] == "1":     # BatchNorm affine (bnX.* / downsample.1.*)
            out[k] = ((0.6 + 0.4 * rs.random_sample(shp)) if k.endswith("weight") else 0.05 * rs.standard_normal(shp)).astype(np.float32)
        else:                                                 # nn.Linear bias
            out[k] = (0.02 * rs.standard_normal(shp)).astype(np.float32)
    return out


def make_image_batch(seed: int, n: int, size: int = 224) -> np.ndarray:
    """[n,3,size,size] fp32 crops, normalised-image-like (zero mean, unit scale, smooth + noise)."""
    rs = np.random.RandomState(seed + 4242)
    yy, xx = np.meshgrid(np.linspace(-1, 1, size), np.linspace(-1, 1, size), indexing="ij")
    imgs = []
    for i in range(n):
        a, b, c = rs.standard_normal(3)
        base = np.stack([np.sin(3 * a * xx + b) * np.cos(2 * c * yy), xx * a - yy * b, np.cos(4 * (xx * yy) + c)], 0)
        imgs.append(base + 0.5 * rs.standard_normal((3, size, size)))
    return np.stack(imgs).astype(np.float32)


def build_synthetic_hmr(seed: int, device="cpu", precision: str = "bf16"):
    """tepose_b200.HMR (ResNet-50 + regressor) of `precision` with make_hmr_state(seed) loaded, on `device`, in eval mode."""
    import tempfile
    import torch
    from .hmr import hmr
    old = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        write_base_data(os.path.join(tmp, "data", "base_data"), seed)      # asset paths are cwd-relative
        os.chdir(tmp)
        try:
            model = hmr(pretrained=False, precision=precision)
        finally:
            os.chdir(old)
    own = model.state_dict()
    sd = make_hmr_state({k: v.shape for k, v in own.items()}, seed)
    for k, v in sd.items():
        own[k] = torch.as_tensor(v)
    model.load_state_dict(own, strict=True)
    return model.to(device).eval()
