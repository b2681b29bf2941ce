"""CPU tests: the oracle against (i) golden vectors produced by the unmodified
reference modules (oracle/make_golden.py), (ii) the independent float64 restatement,
(iii) invariants of the un-pinned smplx boundary (SURVEY.md H9)."""
import os

import numpy as np
import pytest
import torch

from oracle import np64, synth, torch_ref
from tests.helpers import load_forward_golden

GOLD = os.path.join(os.path.dirname(__file__), "golden")
FWD = sorted(f for f in os.listdir(GOLD) if f.startswith("fwd_"))


@pytest.mark.parametrize("fname", FWD)
def test_oracle_matches_reference_golden(fname):
    cfg, gold, cut = load_forward_golden(os.path.join(GOLD, fname))
    sd = synth.make_state_dict(cfg["seed"], cfg["n_layers"], cfg["hidden"])
    m = torch_ref.SmplModel.synthetic(cfg["seed"])
    x = torch.from_numpy(synth.make_input(cfg["seed"], cfg["batch"], cfg["seqlen"]))
    out = cut(torch_ref.tepose_forward(sd, m, x, cfg["n_layers"], cfg["hidden"],
                                       is_train=cfg.get("is_train", False),
                                       J_regressor=m.J_regressor_h36m if cfg.get("use_h36m") else None))
    for k, g in gold.items():
        assert out[k].shape == g.shape
        # same torch ops on the same machine class: tight, but not bitwise across CPUs
        np.testing.assert_allclose(out[k].numpy(), g, atol=2e-5, rtol=1e-5, err_msg=k)


def test_geometry_matches_reference_golden():
    z = np.load(os.path.join(GOLD, "geometry.npz"))
    t = torch.from_numpy
    np.testing.assert_allclose(torch_ref.rot6d_to_rotmat(t(z["x6"])).numpy(), z["rot6d"], atol=1e-6)
    got = torch_ref.rotmat_to_angle_axis(t(z["R"])).numpy()
    np.testing.assert_allclose(got, z["r2aa"], atol=1e-6)
    np.testing.assert_allclose(torch_ref.batch_rodrigues_quat(t(z["aa"])).numpy(), z["rod_q"], atol=1e-6)
    np.testing.assert_allclose(torch_ref.projection(t(z["joints"]), t(z["cam"])).numpy(), z["proj"],
                               rtol=1e-5, atol=1e-4)


def test_np64_geometry_agrees():
    z = np.load(os.path.join(GOLD, "geometry.npz"))
    np.testing.assert_allclose(np64.rot6d_to_rotmat(z["x6"][4:]), z["rot6d"][4:], atol=2e-6)
    for R, aa in zip(z["R"][4:], z["r2aa"][4:]):
        ref = np64.rotmat_to_angle_axis(R)
        # compare as rotations: axis-angle is ill-conditioned near pi
        np.testing.assert_allclose(np64.rodrigues(ref), np64.rodrigues(aa), atol=5e-6)
    got = torch_ref.batch_rodrigues_smplx(torch.from_numpy(z["aa"])).numpy()
    for a, R in zip(z["aa"], got):
        np.testing.assert_allclose(np64.rodrigues(a), R, atol=1e-6)


def test_np64_encoder_and_ief_agree():
    for L, H, B, T in ((1, 32, 2, 4), (2, 24, 2, 3)):
        sd = synth.make_state_dict(5, L, H)
        x = synth.make_input(5, B, T)
        for train in (False, True):
            a = torch_ref.encoder_forward(sd, torch.from_numpy(x), L, H, is_train=train).detach().numpy()
            b = np64.encoder(sd, x, L, H, is_train=train)
            np.testing.assert_allclose(a, b, atol=2e-5)
        feat = np64.encoder(sd, x, L, H)
        p, s, c = torch_ref.ief_forward(sd, torch.from_numpy(feat.astype(np.float32)))
        p64, s64, c64 = np64.ief(sd, feat)
        np.testing.assert_allclose(p.numpy(), p64, atol=1e-5)
        np.testing.assert_allclose(s.numpy(), s64, atol=1e-5)
        np.testing.assert_allclose(c.numpy(), c64, atol=1e-5)


def test_smpl_restatement_float64_crosscheck():
    model, extra = synth.make_smpl_model(3), synth.make_extra_regressors(3)
    m = torch_ref.SmplModel(model, extra)
    bodies = synth.make_bodies(3, 3)
    betas = torch.from_numpy(bodies["betas"])
    verts, joints, R = torch_ref.smpl_forward(m, betas, pose_aa=torch.from_numpy(bodies["pose_aa"]))
    for i in range(3):
        R64 = np.stack([np64.rodrigues(a) for a in bodies["pose_aa"][i].reshape(24, 3)])
        v64, j64, _ = np64.smpl(model, extra, bodies["betas"][i], R64,
                                torch_ref.JOINT_SOURCE_49, synth.SMPL_EXTRA_VERTEX_IDS)
        np.testing.assert_allclose(verts[i].numpy(), v64, atol=2e-5)
        np.testing.assert_allclose(joints[i].numpy(), j64, atol=2e-5)
        kp = torch_ref.projection(joints[i:i + 1], torch.from_numpy(bodies["cam"][i:i + 1]))[0].numpy()
        np.testing.assert_allclose(kp, np64.projection(j64, bodies["cam"][i].astype(np.float64)), atol=2e-3)


def test_smpl_invariants():
    """H9: identity pose => verts == v_shaped and joints == J_regressor @ v_shaped;
    a global rotation rotates the mesh rigidly about the root joint; skinning weights
    are a partition of unity."""
    m = torch_ref.SmplModel.synthetic(4, dtype=torch.float64)
    betas = torch.from_numpy(synth.make_bodies(4, 2)["betas"]).double()
    eye = torch.eye(3, dtype=torch.float64).expand(2, 24, 3, 3).contiguous()
    verts, posed = torch_ref.smpl_lbs(m, betas, eye)
    v_shaped = m.v_template[None] + torch.einsum("bl,mkl->bmk", betas, m.shapedirs)
    assert torch.allclose(verts, v_shaped, atol=1e-12)
    assert torch.allclose(posed, torch.einsum("bik,ji->bjk", v_shaped, m.J_regressor), atol=1e-12)
    assert torch.allclose(m.lbs_weights.sum(1), torch.ones(6890, dtype=torch.float64), atol=1e-6)
    Rg = torch.from_numpy(np64.rodrigues(np.array([0.3, -0.5, 0.2])))
    R = eye.clone()
    R[:, 0] = Rg
    v_rot, _ = torch_ref.smpl_lbs(m, betas, R)
    root = posed[:, 0:1]
    assert torch.allclose(v_rot, (verts - root) @ Rg.T + root, atol=1e-7)  # weights sum to 1 within fp32 eps


def test_causal_state_identity():
    """SURVEY.md F3: the encoder equals three causal pieces (L=1)."""
    sd = synth.make_state_dict(6, 1, 48)
    x = torch.from_numpy(synth.make_input(6, 3, 7))
    full = torch_ref.encoder_forward(sd, x, 1, 48)
    hF, hB, hS = torch_ref.encoder_causal_states(sd, x, 48)
    assert torch.allclose(torch_ref.encoder_from_states(sd, hF, hB, hS), full, atol=1e-5)
    # carried state over two chunks == one pass
    hF1, hB1, _ = torch_ref.encoder_causal_states(sd, x[:, :4], 48)
    hF2, hB2, hS2 = torch_ref.encoder_causal_states(sd, x[:, 4:], 48, h0=(hF1, hB1))
    assert torch.allclose(hF2, hF, atol=1e-5) and torch.allclose(hB2, hB, atol=1e-5)
    assert torch.allclose(hS2, hS, atol=1e-6)
