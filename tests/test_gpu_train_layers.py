"""Training of multi-layer encoders (the released configuration is L = 2, H = 1024, T = 6): the oracle pinned to the reference at
L = 2, the product's train-mode forward against that golden, and the hand-written backward through stacked GRU layers against
torch.autograd through the oracle's nn.GRU(num_layers=L)."""
import os

import numpy as np
import pytest
import torch

from oracle import synth, train_ref
from tests.helpers import build_product_model, compare_outputs, load_forward_golden

DEV = "cuda:0"
GOLDEN_L2 = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fwd_L2_H96_B1_T3_train.npz")


def identity_masks(n_rows):
    """Keep masks of 0.5: a * mask / (1 - p) is the identity, i.e. the reference's train-mode forward with dropout inactive."""
    return np.full((train_ref.N_ITER, 2, n_rows, 1024), 0.5, dtype=np.float32)


def rel_err(got, ref):
    ref = torch.as_tensor(ref).double()
    return float((got.detach().cpu().double() - ref).abs().max() / (ref.abs().max() + 1e-30))


def test_train_oracle_reproduces_two_layer_golden():
    """The golden holds the unmodified reference's outputs for is_train=True with dropout inactive at L = 2."""
    cfg, gold, _ = load_forward_golden(GOLDEN_L2)
    seed, B, T, L, H = cfg["seed"], cfg["batch"], cfg["seqlen"], cfg["n_layers"], cfg["hidden"]
    assert (seed, B, T, L, H) == (15, 1, 3, 2, 96)
    sd = synth.make_state_dict(seed, L, H)
    orc = train_ref.TrainOracle(sd, seed, L, H)
    assert isinstance(orc.gru_fwd, torch.nn.GRU) and orc.gru_fwd.num_layers == 2 and orc.gru_rec.num_layers == 2
    x = synth.make_input(seed, B, T)
    out = orc.forward(torch.as_tensor(x), torch.as_tensor(identity_masks(2 * B)))
    compare_outputs(out, gold, label="oracle L2 train")
    # torch.autograd reaches every GRU tensor of both layers, except the top layer's gru_rec.weight_hh (one step from h_0 = 0)
    _, _, grads = orc.loss_and_grads(x, identity_masks(2 * B), train_ref.make_targets(seed, 2 * B))
    for name, g in grads.items():
        if name == "encoder.gru_rec.weight_hh_l1":
            assert float(g.abs().max()) == 0.0
        elif ".gru_" in name:
            assert float(g.abs().max()) > 0.0, name


@pytest.mark.parametrize("L", [1, 2, 3])
def test_path_parameters_cover_every_trained_parameter(L):
    from tepose_b200.train import path_parameters
    model, _ = build_product_model(7, 4, L, 64)
    want = [n for n, _ in model.named_parameters() if not n.startswith("regressor.smpl.")]
    assert [n for n, _ in path_parameters(model)] == want
    assert len([n for n in want if ".gru_" in n]) == 12 * L


# ------------------------------------------------------------------------------------------------------------ GPU
def train_step(model, x, masks, tgt):
    out = model(torch.from_numpy(x).to(DEV), is_train=True, dropout_masks=torch.from_numpy(masks).to(DEV))[-1]
    loss = train_ref.synthetic_loss(out, tgt)
    loss.backward()
    return out, loss


@pytest.mark.gpu
def test_train_mode_forward_reproduces_two_layer_golden():
    cfg, gold, _ = load_forward_golden(GOLDEN_L2)
    seed, B, T, L, H = cfg["seed"], cfg["batch"], cfg["seqlen"], cfg["n_layers"], cfg["hidden"]
    model, _ = build_product_model(seed, T, L, H, "fp32", DEV)
    model.train()
    x = torch.from_numpy(synth.make_input(seed, B, T)).to(DEV)
    out = model(x, is_train=True, dropout_masks=torch.from_numpy(identity_masks(2 * B)).to(DEV))[-1]
    assert out["verts"].requires_grad
    print(compare_outputs(out, gold, label="train-mode L2"))


def check_fp32_gradients(seed, L, B, T, H, show=0):
    """The bar of the L = 1 training step: loss within 1e-4 relative, outputs within the inference tolerances, every parameter
    gradient within 1e-4 max-norm relative of torch.autograd through the oracle."""
    model, sd = build_product_model(seed, T, L, H, "fp32", DEV)
    model.train()
    x = synth.make_input(seed, B, T)
    masks = train_ref.make_masks(seed, 2 * B)
    tgt = train_ref.make_targets(seed, 2 * B)
    out, loss = train_step(model, x, masks, tgt)
    ref_out, ref_loss, ref_grads = train_ref.TrainOracle(sd, seed, L, H).loss_and_grads(x, masks, tgt)
    assert abs(float(loss.detach()) - ref_loss) < 1e-4 * max(1.0, abs(ref_loss))
    for k in ("kp_2d", "kp_3d", "rotmat", "verts"):
        assert float((out[k].detach().cpu() - ref_out[k]).abs().max()) < (1e-3 if k == "kp_2d" else 1e-4), k
    params = dict(model.named_parameters())
    assert sorted(ref_grads) == sorted(n for n in params if not n.startswith("regressor.smpl."))
    worst = {}
    for name, g_ref in ref_grads.items():
        assert params[name].grad is not None, name
        worst[name] = rel_err(params[name].grad, g_ref)
    if show:
        print(f"L={L} B={B} T={T} H={H} worst gradient errors (max-norm relative):",
              {k: f"{v:.1e}" for k, v in sorted(worst.items(), key=lambda kv: -kv[1])[:show]})
    bad = {k: v for k, v in worst.items() if v > 1e-4}
    assert not bad, bad
    assert all(p.grad is None for n, p in params.items() if n.startswith("regressor.smpl."))
    # the top layer's gru_rec forward direction is one step from h_0 = 0; the directions below it are full (with T = 1 every
    # direction is one step from h_0 = 0, and no gradient reaches any weight_hh)
    assert float(params[f"encoder.gru_rec.weight_hh_l{L - 1}"].grad.abs().max()) == 0.0
    for l in range(L - 1):
        for name in (f"encoder.gru_rec.weight_hh_l{l}", f"encoder.gru_rec.weight_hh_l{l}_reverse", f"encoder.gru_fwd.weight_hh_l{l}"):
            assert (float(params[name].grad.abs().max()) > 0.0) == (T > 1), name


@pytest.mark.gpu
@pytest.mark.parametrize("seed,L,B,T,H", [(61, 2, 2, 5, 64), (62, 2, 3, 1, 96), (63, 2, 2, 2, 128), (64, 3, 2, 4, 64)])
def test_multi_layer_train_step_gradients_match_oracle(seed, L, B, T, H):
    check_fp32_gradients(seed, L, B, T, H)


@pytest.mark.gpu
def test_released_configuration_train_step_gradients_match_oracle():
    """B = 32, T = 6, L = 2, H = 1024, fp32: every parameter gradient against torch.autograd through the oracle on the CPU."""
    check_fp32_gradients(0, 2, 32, 6, 1024, show=6)


@pytest.mark.gpu
@pytest.mark.parametrize("tc", [False, True])
def test_two_layer_mixed_precision_gradients_are_close(tc):
    """precision='bf16', L = 2: the bars of the L = 1 mixed-precision step -- 1e-2 max-norm relative downstream of the encoder,
    cosine >= 0.97 on every GRU tensor, the lower layer's included."""
    seed, B, T, H = 65, 4, 6, 256
    model, sd = build_product_model(seed, T, 2, H, "bf16", DEV)
    model.train()
    model.train_tensor_core_grads = tc
    x = synth.make_input(seed, B, T)
    masks = train_ref.make_masks(seed, 2 * B)
    tgt = train_ref.make_targets(seed, 2 * B)
    train_step(model, x, masks, tgt)
    _, _, ref_grads = train_ref.TrainOracle(sd, seed, 2, H).loss_and_grads(x, masks, tgt)
    params = dict(model.named_parameters())
    cosines = {}
    for name, g_ref in ref_grads.items():
        g = params[name].grad.detach().cpu().double().reshape(-1)
        r = g_ref.double().reshape(-1)
        if float(r.abs().max()) == 0.0:
            assert float(g.abs().max()) == 0.0, name
            continue
        if ".gru_" in name:
            cosines[name] = float((g * r).sum() / (g.norm() * r.norm() + 1e-30))
        else:
            assert rel_err(params[name].grad, g_ref) < 1e-2, (name, rel_err(params[name].grad, g_ref))
    print("lowest GRU cosines:", {k: f"{v:.4f}" for k, v in sorted(cosines.items(), key=lambda kv: kv[1])[:6]})
    assert any(k.endswith("_l0") for k in cosines) and any(k.endswith("_l1") for k in cosines)
    bad = {k: v for k, v in cosines.items() if v < 0.97}
    assert not bad, bad
