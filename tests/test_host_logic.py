"""CPU tests of the Python host layer (packing, segment tables, job time-indexing, joint
composition, state_dict compatibility) with the native calls emulated on CPU
(tests/fake_native.py).  The CUDA kernels themselves are tested in the -m gpu files."""
import os

import numpy as np
import pytest
import torch

from oracle import synth, torch_ref
from tests import fake_native
from tests.helpers import base_data_cwd, build_product_model, compare_outputs, load_forward_golden, oracle_forward

GOLD = os.path.join(os.path.dirname(__file__), "golden")
CASES = [
    dict(seed=21, batch=2, seqlen=4, n_layers=1, hidden=64),
    dict(seed=22, batch=3, seqlen=5, n_layers=2, hidden=64),
    dict(seed=23, batch=2, seqlen=3, n_layers=3, hidden=32),
    dict(seed=24, batch=2, seqlen=6, n_layers=1, hidden=96, use_h36m=True),
    dict(seed=25, batch=2, seqlen=4, n_layers=2, hidden=32, is_train=True),
    dict(seed=26, batch=1, seqlen=1, n_layers=1, hidden=32),
]


@pytest.mark.parametrize("cfg", CASES, ids=lambda c: "L{n_layers}_H{hidden}_B{batch}_T{seqlen}".format(**c))
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_host_schedule_matches_oracle(cfg, precision):
    model, sd = build_product_model(cfg["seed"], cfg["seqlen"], cfg["n_layers"], cfg["hidden"], precision)
    x = synth.make_input(cfg["seed"], cfg["batch"], cfg["seqlen"])
    ref, m = oracle_forward(cfg["seed"], sd, x, cfg["n_layers"], cfg["hidden"], cfg.get("is_train", False),
                            cfg.get("use_h36m", False))
    with fake_native.install() as fake:
        out = model(torch.from_numpy(x), is_train=cfg.get("is_train", False),
                    J_regressor=m.J_regressor_h36m if cfg.get("use_h36m") else None)[-1]
    if precision == "fp32":
        compare_outputs(out, ref, label=str(cfg))
    else:   # bf16 operands in K1/K2: <= 1 mm on the mesh (north_star), rotations loosely
        compare_outputs(out, ref, vert_tol=1e-3, rot_tol=2e-3, kp2d_tol=5e-2, label=str(cfg))
    kinds = [c[0] for c in fake.calls]
    assert kinds.count("gru") == cfg["n_layers"]
    assert ("gemm_bf16_tc" in kinds) == (precision == "bf16")


def test_single_step_direction_is_not_run_for_T_steps():
    """SURVEY.md F3: for the last layer gru_rec's forward direction needs ONE step."""
    model, _ = build_product_model(31, 8, 1, 32)
    with fake_native.install() as fake:
        model(torch.from_numpy(synth.make_input(31, 2, 8)))
    gru = [c for c in fake.calls if c[0] == "gru"][0]
    assert gru[5] == [8, 8, 1]


def test_state_dict_keys_match_reference_layout():
    """SURVEY.md App. A.1: released checkpoints must load with strict=True."""
    model, _ = build_product_model(32, 4, 2, 32)
    keys = set(model.state_dict().keys())
    expect = set(synth.make_state_dict(0, 2, 32).keys())
    assert expect <= keys
    smpl_keys = {k for k in keys if k.startswith("regressor.smpl.")}
    assert smpl_keys == {"regressor.smpl." + n for n in (
        "faces_tensor", "v_template", "shapedirs", "J_regressor", "posedirs", "parents", "lbs_weights",
        "vertex_joint_selector.extra_joints_idxs", "betas", "global_orient", "body_pose", "J_regressor_extra")}
    assert keys - expect - smpl_keys == set()
    assert model.state_dict()["regressor.smpl.betas"].shape == (64, 10)
    assert "joint_map" not in " ".join(keys)


@pytest.mark.parametrize("fname", sorted(f for f in os.listdir(GOLD) if f.startswith("fwd_")))
def test_host_layer_against_reference_golden(fname):
    cfg, gold, cut = load_forward_golden(os.path.join(GOLD, fname))
    model, sd = build_product_model(cfg["seed"], cfg["seqlen"], cfg["n_layers"], cfg["hidden"])
    x = synth.make_input(cfg["seed"], cfg["batch"], cfg["seqlen"])
    m = torch_ref.SmplModel.synthetic(cfg["seed"])
    with fake_native.install():
        out = model(torch.from_numpy(x), is_train=cfg.get("is_train", False),
                    J_regressor=m.J_regressor_h36m if cfg.get("use_h36m") else None)[-1]
    compare_outputs(cut(out), gold, label=fname)


def test_smpl_module_api():
    import tepose_b200
    with base_data_cwd(5):
        smpl = tepose_b200.SMPL(tepose_b200.SMPL_MODEL_DIR, batch_size=2, create_transl=False)
    bodies = synth.make_bodies(5, 3)
    m = torch_ref.SmplModel.synthetic(5)
    aa = torch.from_numpy(bodies["pose_aa"])
    betas = torch.from_numpy(bodies["betas"])
    with fake_native.install():
        out = smpl(betas=betas, body_pose=aa[:, 3:], global_orient=aa[:, :3], pose2rot=True)
        R = torch_ref.batch_rodrigues_smplx(aa.reshape(-1, 3)).reshape(3, 24, 3, 3)
        out2 = smpl(betas=betas, body_pose=R[:, 1:], global_orient=R[:, :1], pose2rot=False)
    v, j, _ = torch_ref.smpl_forward(m, betas, pose_aa=aa)
    assert out.vertices.shape == (3, 6890, 3) and out.joints.shape == (3, 49, 3)
    assert torch.allclose(out.vertices, v, atol=1e-5) and torch.allclose(out.joints, j, atol=1e-5)
    assert torch.allclose(out2.vertices, v, atol=1e-5) and torch.allclose(out2.joints, j, atol=1e-5)
    assert smpl.faces.shape == (13776, 3)
    assert tepose_b200.JOINT_MAP["OP Nose"] == 24 and len(tepose_b200.JOINT_NAMES) == 49
    assert tepose_b200.H36M_TO_J14 == [6, 5, 4, 1, 2, 3, 16, 15, 14, 11, 12, 13, 8, 10]


def test_train_mode_refuses_loudly():
    model, _ = build_product_model(33, 3, 1, 32)
    model.train()
    with fake_native.install(), pytest.raises(NotImplementedError):
        model(torch.from_numpy(synth.make_input(33, 1, 3)))


def test_cpu_tensor_is_rejected_without_fallback():
    model, _ = build_product_model(34, 3, 1, 32)
    with pytest.raises(RuntimeError, match="no CPU path|CUDA"):
        model(torch.from_numpy(synth.make_input(34, 1, 3)))


def test_live_stream_matches_causal_oracle():
    """Carried-state live mode against torch.nn.GRU stepped with explicit h0 (SURVEY.md F4)."""
    from tepose_b200.live import LiveTePose
    seed, H, B, N = 41, 64, 2, 5
    model, sd = build_product_model(seed, 16, 1, H)
    m = torch_ref.SmplModel.synthetic(seed)
    feats = torch.from_numpy(synth.make_input(seed, B, N))[:, :, :2048]
    with fake_native.install():
        live = LiveTePose(model, batch=B, use_graph=False)
        outs = [{k: v.clone() for k, v in live.step(feats[:, t]).items()} for t in range(N)]
    # oracle: feed frames in order, each committed with its own predicted theta
    hF = hB = None
    prev = None
    for t in range(N):
        newest = torch.cat([feats[:, t], torch.zeros(B, 85)], dim=1)[:, None]
        if prev is None:
            hFt, hBt, hS = torch_ref.encoder_causal_states(sd, newest, H)
        else:
            hFc, hBc, _ = torch_ref.encoder_causal_states(sd, prev, H, h0=None if hF is None else (hF, hB))
            hF, hB = hFc, hBc
            hFt, hBt, hS = torch_ref.encoder_causal_states(sd, newest, H, h0=(hF, hB))
        feat = torch_ref.encoder_from_states(sd, hFt, hBt, hS)
        ref = torch_ref.regressor_forward(sd, m, feat)
        compare_outputs(outs[t], ref, label=f"live frame {t}")
        prev = torch.cat([feats[:, t], ref["theta"]], dim=1)[:, None]


# ------------------------------------------------------------------------------------------------ folded heads + IEF
def test_ief_closed_form_equals_the_loop_in_float64():
    """Regressor.folded(): n IEF iterations == A^n p0 + S_n (Q f + c) (no nonlinearity: lib/models/spin.py:250-261)."""
    from oracle import np64
    model, sd = build_product_model(45, 4, 1, 32)
    reg = model.regressor
    feat = np.random.Generator(np.random.PCG64(9)).standard_normal((3, 2048))
    for n_iter in (1, 3, 4):
        fd = reg.folded(n_iter)
        p0 = np.zeros(160)
        p0[:144] = sd["regressor.init_pose"][0]; p0[144:154] = sd["regressor.init_shape"][0]; p0[154:157] = sd["regressor.init_cam"][0]
        got = feat @ fd["G64"].numpy().T + fd["g64"].numpy() + fd["An64"].numpy() @ p0
        pose, shape, cam = np64.ief(sd, feat, n_iter)
        want = np.concatenate([pose, shape, cam], axis=1)
        np.testing.assert_allclose(got[:, :157], want, atol=1e-12, rtol=1e-10)
        assert np.all(got[:, 157:] == 0)


@pytest.mark.parametrize("cfg", CASES[:4], ids=lambda c: "L{n_layers}_H{hidden}_B{batch}_T{seqlen}".format(**c))
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_folded_path_matches_oracle(cfg, precision):
    model, sd = build_product_model(cfg["seed"], cfg["seqlen"], cfg["n_layers"], cfg["hidden"], precision)
    model.fold_linear = True
    x = synth.make_input(cfg["seed"], cfg["batch"], cfg["seqlen"])
    ref, m = oracle_forward(cfg["seed"], sd, x, cfg["n_layers"], cfg["hidden"], False, cfg.get("use_h36m", False))
    with fake_native.install() as fake:
        out = model(torch.from_numpy(x), J_regressor=m.J_regressor_h36m if cfg.get("use_h36m") else None)[-1]
        feat = torch.from_numpy(np.random.Generator(np.random.PCG64(4)).standard_normal((5, 2048)).astype(np.float32))
        a = model.regressor.forward_folded(feat)[-1]
        b = model.regressor(feat)[-1]
    kinds = [c[0] for c in fake.calls]
    first_smpl = kinds.index("smpl")
    assert "heads_cat" not in kinds[:first_smpl]                 # one GEMM replaced the heads and the IEF layers
    assert ("gemm_f32", cfg["batch"], 160, 3 * cfg["hidden"]) in fake.calls
    if precision == "fp32":
        compare_outputs(out, ref, label=str(cfg))
    else:
        compare_outputs(out, ref, vert_tol=1e-3, rot_tol=2e-3, kp2d_tol=5e-2, label=str(cfg))
    compare_outputs(a, b, label="regressor folded vs loop", **({} if precision == "fp32" else dict(vert_tol=1e-3, rot_tol=2e-3, kp2d_tol=5e-2)))


def test_large_batches_run_as_balanced_groups():
    """bf16 mode, B > 32: the encoder + heads/IEF run per group of <= 32 sequences (their fast kernels hold one 32-row
    tile), the SMPL pass once over all rows; results must not depend on the grouping."""
    cfg = dict(seed=27, batch=70, seqlen=3, n_layers=1, hidden=32)
    model, sd = build_product_model(cfg["seed"], cfg["seqlen"], cfg["n_layers"], cfg["hidden"], "bf16")
    x = synth.make_input(cfg["seed"], cfg["batch"], cfg["seqlen"])
    ref, m = oracle_forward(cfg["seed"], sd, x, cfg["n_layers"], cfg["hidden"])
    with fake_native.install() as fake:
        out = model(torch.from_numpy(x))[-1]
    compare_outputs(out, ref, vert_tol=1e-3, rot_tol=2e-3, kp2d_tol=5e-2, label="grouped")
    grus = [c for c in fake.calls if c[0] == "gru"]
    assert [c[2] for c in grus] == [24, 24, 22]                    # balanced groups of the 70 sequences
    assert [c[0] for c in fake.calls].count("smpl") == 1 and out["verts"].shape[0] == 70


def test_device_guard_is_transparent_without_cuda_tensors():
    """nv.device_guard (ADVICE r1: every public entry point runs with its tensors' device current) must not touch CUDA when no
    CUDA tensor is involved, and must keep signature / return value."""
    import tepose_b200._native as nv
    calls = []

    @nv.device_guard
    def f(a, b=2):
        calls.append((a, b))
        return a

    t = torch.zeros(2)
    assert f(t, b=3) is t and calls == [(t, 3)]
    assert f.__name__ == "f"
