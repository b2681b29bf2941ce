"""The mixed-precision training step (precision='bf16', with and without tensor-core weight gradients) against float64 on its
own operands, stage by stage, at the shapes bench.py reports and at the shapes where the kernels change path.

The end-to-end tests of test_gpu_train.py / test_gpu_train_layers.py compare the bf16 step with the fp32 oracle, and can only
ask for cosine >= 0.97 on the GRU gradients: the bf16 forward moves the states by ~1e-3 and flips relu masks.  Here every stage
is teacher-forced on what the product itself saved or computed, so the bars are near fp32 level:
  - forward: every step of every job against a float64 GRU cell fed the product's saved fp32 input and state, rounded to
    bf16 where the kernels round them (bf16(x) . bf16(W_ih)^T, bf16(h) . bf16(W_hh)^T);
  - BPTT: the cell adjoint replayed in float64 from the captured dL/dh of the heads (top layer) or from the captured upper
    d_gi . W_ih (lower layers), with the per-step d_gh . W_hh on the product's own d_gh, rounded to bf16, and bf16(W_hh);
  - gradients: every weight-gradient GEMM, the heads' weight gradients and every bias gradient (column sum) under gemm_check
    on their exact operands, the regressor against the fp32 oracle;
  - controls: a reference without the bf16 rounding exceeds each stage's bound, so the bounds are tighter than bf16.
The step's operands are captured by wrapping train._train_backward, _Ops.weight_grad and _Ops.colsum (monkeypatch): the
product runs unchanged.  Every torch.empty of tepose.py and train.py returns NaN in these runs, so a store a kernel skips
(ragged batch rows, reduction padding) reads back as NaN."""
import math

import pytest
import torch

import tepose_b200.tepose as tepose_mod
import tepose_b200._native as nv
from oracle import synth, train_ref
from tepose_b200 import train as tr
from tests.helpers import build_product_model, gemm_check

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# (seed, L, H, B, T)
SHAPES = [
    (80, 1, 2048, 32, 16),     # BASELINE configs[4] as bench.py runs it: k_gru_umma, skinny M=32 K=6144, dW_hh reduction 480 -> 512
    (81, 2, 1024, 32, 6),      # released configuration: three full lower directions on k_gru_umma, reduction 160 -> 192
    (82, 1, 256, 5, 4),        # ragged batch rows in the umma gate stores
    (83, 1, 128, 40, 3),       # B > 32: the generic k_gru_bf16 forward with gates, skinny at M = 40
    (84, 2, 96, 2, 5),         # H % 128 != 0: generic kernels at every layer
    (85, 1, 128, 3, 1),        # every direction one step from zero, no dW_hh
]
SHAPE_IDS = ["L1-H2048-B32-T16", "L2-H1024-B32-T6", "L1-H256-B5-T4", "L1-H128-B40-T3", "L2-H96-B2-T5", "L1-H128-B3-T1"]

# Bars, a few times above the worst case measured on an NVIDIA B200 (1000 W power limit) over every shape x tc
FWD_ABS = 4e-5             # r, z, n, h_t: absolute (measured 9.5e-6)
FWD_GHN = 1e-5             # gh_n: max-abs error over max |gh_n| of the step (measured 1.5e-6)
BPTT_REL = 1e-5            # d_gi, d_gh: max-abs error over max |ref| per job and step (measured 1.0e-6)
REGRESSOR_REL = 1e-2       # regressor gradients against the fp32 oracle (max-norm relative), the bar of test_gpu_train.py


class _NaNTorch:
    """The `torch` a product module sees: `empty` returns NaN-filled tensors."""

    def __getattr__(self, name):
        return getattr(torch, name)

    @staticmethod
    def empty(*size, **kw):
        t = torch.empty(*size, **kw)
        return t.fill_(float("nan")) if t.is_floating_point() else t


def bf(t):
    """float64 copy of RN_bf16(t): the operand a bf16 kernel reads."""
    return t.to(torch.bfloat16).double()


def amax(t):
    """max |t|, with NaN as inf (Python's max() would drop a NaN)."""
    v = float(t.abs().max())
    return math.inf if math.isnan(v) else v


def rel(got, ref):
    return amax(got.double() - ref) / (amax(ref) + 1e-30)


# ------------------------------------------------------------------------------------------------------------- indexing
# The step-index conventions of train.py's backward (t_in / t_out, shared with the fp32 path, which test_gpu_train_layers.py
# holds to torch.autograd at 1e-4), restated: "f" = gru_fwd, "b" = gru_rec reverse, "s" = gru_rec forward (one step in the
# top layer).  Gates are indexed like the direction's output (t_out), states in run order, d_gi rows by t_in, d_gh rows by s.
def pname(l, d, k):
    return f"encoder.gru_fwd.{k}_l{l}" if d == "f" else f"encoder.gru_rec.{k}_l{l}" + ("_reverse" if d == "b" else "")


def t_in(l, d, s, top, T):
    if d == "f":
        return s
    if d == "b":
        return s if l == 0 else T - 1 - s
    if l == top:
        return T - 1 if l == 0 else 0
    return T - 1 - s if l == 0 else s


def t_out(l, d, s, top, T):
    return T - 1 - s if d == "b" and l != top else s


def jobs_of(L):
    """(layer, direction) in the order the backward visits them (colsum and dW_ih calls)."""
    return [(l, d) for l in range(L - 1, -1, -1) for d in ("f", "b", "s")]


# ------------------------------------------------------------------------------------------------------------- capture
class Step:
    """One training step of a product model with its operands captured."""

    def __init__(self, seed, L, H, B, T, tc, fp32_bptt=False, precision="bf16"):
        self.seed, self.L, self.H, self.B, self.T, self.tc = seed, L, H, B, T, tc
        self.top = L - 1
        model, sd = build_product_model(seed, T, L, H, precision, DEV)
        model.train()
        model.train_tensor_core_grads = tc
        model.train_fp32_bptt = fp32_bptt
        model._debug_capture = dbg = {}
        wg, cs, sv_cap = [], [], {}
        orig_bw, orig_wg, orig_cs = tr._train_backward, tr._Ops.weight_grad, tr._Ops.colsum

        def backward(model_, sv, *g_out):
            sv_cap["layers"] = [{k: {d: t.clone() for d, t in lay[k].items()} for k in ("x", "seq", "gates")} for lay in sv["layers"]]
            sv_cap["h_cat"] = sv["h_cat"].clone()
            return orig_bw(model_, sv, *g_out)

        def weight_grad(g, x, out, rows, tensor_core=False):
            n_out, k_in = out.shape
            rec = {"g": g[:rows, :n_out].clone(), "x": x[:rows, :k_in].clone(), "rows": rows, "tensor_core": tensor_core}
            res = orig_wg(g, x, out, rows, tensor_core=tensor_core)
            rec["out"] = out.clone()
            wg.append(rec)
            return res

        def colsum(a, rows=None, cols=None):
            out = orig_cs(a, rows, cols)
            rows = a.shape[0] if rows is None else rows
            cols = a.shape[1] if cols is None else cols
            cs.append({"a": a[:rows, :cols].clone(), "out": out.clone()})
            return out

        x = synth.make_input(seed, B, T)
        masks = train_ref.make_masks(seed, 2 * B)
        tgt = train_ref.make_targets(seed, 2 * B)
        with pytest.MonkeyPatch.context() as mp:
            mp.setattr(tr, "_train_backward", backward)
            mp.setattr(tr._Ops, "weight_grad", staticmethod(weight_grad))
            mp.setattr(tr._Ops, "colsum", staticmethod(colsum))
            mp.setattr(tr, "torch", _NaNTorch())
            mp.setattr(tepose_mod, "torch", _NaNTorch())
            out = model(torch.from_numpy(x).to(DEV), is_train=True, dropout_masks=torch.from_numpy(masks).to(DEV))[-1]
            train_ref.synthetic_loss(out, tgt).backward()
        torch.cuda.synchronize()
        self.sd, self.x, self.masks, self.tgt = sd, x, masks, tgt
        self.layers, self.h_cat, self.g_hcat, self.g_feat = sv_cap["layers"], sv_cap["h_cat"], dbg["g_hcat"], dbg["g_feat"]
        self.params = {n: p.detach().clone() for n, p in model.named_parameters() if ".gru_" in n}
        self.grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
        self.wg, self.cs = wg, cs
        # colsum calls: fc1, fc2, dec, linear_fwd, linear_rec biases, then (d_gh, d_gi) of every job
        jobs = jobs_of(L)
        assert len(cs) == 5 + 2 * len(jobs), len(cs)
        self.dgh = {j: cs[5 + 2 * i]["a"] for i, j in enumerate(jobs)}
        self.dgi = {j: cs[6 + 2 * i]["a"] for i, j in enumerate(jobs)}
        self.cs_names = ["regressor.fc1.bias", "regressor.fc2.bias", "regressor.dec*.bias", "encoder.linear_fwd.bias",
                         "encoder.linear_rec.bias"]
        for j in jobs:
            self.cs_names += [pname(*j, "bias_hh"), pname(*j, "bias_ih")]
        # weight_grad calls: fc1 (features, IEF state), fc2, dec*, then dW_hh of every full job (T > 1), then dW_ih of every job
        hh = [j for j in jobs if not (j[0] == self.top and j[1] == "s")] if T > 1 else []
        self.wg_names = ["regressor.fc1.weight[:, :2048]", "regressor.fc1.weight[:, 2048:]", "regressor.fc2.weight", "regressor.dec*.weight"]
        self.wg_names += [pname(*j, "weight_hh") for j in hh] + [pname(*j, "weight_ih") for j in jobs]
        assert len(wg) == len(self.wg_names), (len(wg), self.wg_names)
        for rec, name in zip(wg[4:], self.wg_names[4:]):
            l, d = self.job_of(name)
            if "weight_hh" in name:        # d_gh of steps 1..T-1 against the states of steps 0..T-2
                assert torch.equal(rec["g"], self.dgh[(l, d)][B:]), name
                assert torch.equal(rec["x"], self.layers[l]["seq"][d].reshape(T * B, H)[:(T - 1) * B]), name
            else:
                assert torch.equal(rec["g"], self.dgi[(l, d)]), name
            assert torch.equal(rec["out"], self.grads[name]), name
            assert rec["tensor_core"] == tc, name

    def job_of(self, name):
        l = int(name.split("_l")[1][0])
        return l, ("f" if "gru_fwd" in name else ("b" if "_reverse" in name else "s"))


_STEPS = {}


def step(seed, L, H, B, T, tc, fp32_bptt=False):
    key = (seed, L, H, B, T, tc, fp32_bptt)
    if key not in _STEPS:
        _STEPS[key] = Step(seed, L, H, B, T, tc, fp32_bptt)
    return _STEPS[key]


_ORACLE = {}


def oracle_grads(c):
    key = (c.seed, c.L, c.H, c.B, c.T)
    if key not in _ORACLE:
        _ORACLE.clear()
        _ORACLE[key] = train_ref.TrainOracle(c.sd, c.seed, c.L, c.H).loss_and_grads(c.x, c.masks, c.tgt)[2]
    return _ORACLE[key]


# ------------------------------------------------------------------------------------------------------------- references
def forward_errors(c, rnd=bf):
    """Worst errors of the saved gates [r | z | n | gh_n] and states against a float64 GRU cell teacher-forced on the saved
    fp32 input and previous state, per job.  rnd: the rounding of the matmul operands (bf16 as the kernels read them)."""
    B, T, H, top = c.B, c.T, c.H, c.top
    worst = {}
    for l in range(c.L):
        for d in ("f", "b", "s"):
            single = l == top and d == "s"
            w_ih, b_ih = c.params[pname(l, d, "weight_ih")], c.params[pname(l, d, "bias_ih")].double()
            w_hh, b_hh = rnd(c.params[pname(l, d, "weight_hh")]), c.params[pname(l, d, "bias_hh")].double()
            x_in = c.layers[l]["x"]["f" if d == "f" else "r"][:, :w_ih.shape[1]]
            gi_all = rnd(x_in) @ rnd(w_ih).T + b_ih
            gates = c.layers[l]["gates"][d]
            seq = None if single else c.layers[l]["seq"][d]
            e = {"r": 0.0, "z": 0.0, "n": 0.0, "h": 0.0, "gh_n": 0.0}
            for s in range(1 if single else T):
                ti = t_in(l, d, s, top, T)
                gi = gi_all[ti * B:(ti + 1) * B]
                hp = None if s == 0 else seq[s - 1].double()
                gh = b_hh.expand(B, -1) if hp is None else rnd(seq[s - 1]) @ w_hh.T + b_hh
                r = torch.sigmoid(gi[:, :H] + gh[:, :H])
                z = torch.sigmoid(gi[:, H:2 * H] + gh[:, H:2 * H])
                n = torch.tanh(gi[:, 2 * H:] + r * gh[:, 2 * H:])
                h = (1 - z) * n + (0.0 if hp is None else z * hp)
                got = gates[0 if single else t_out(l, d, s, top, T)].double()
                h_got = c.h_cat[:, H:2 * H] if single else seq[s]
                for k, ref, g in (("r", r, got[:, :H]), ("z", z, got[:, H:2 * H]), ("n", n, got[:, 2 * H:3 * H]), ("h", h, h_got.double())):
                    e[k] = max(e[k], amax(g - ref))
                e["gh_n"] = max(e["gh_n"], rel(got[:, 3 * H:], gh[:, 2 * H:]))
            worst[(l, d)] = e
    return worst


def bptt_errors(c, whh="bf16", dgh_bf16=True):
    """Per (job, step): max-norm relative errors of the captured d_gi and d_gh against the cell adjoint replayed in float64
    (the formulas test_gpu_train.py::test_gru_cell_backward_matches_autograd pins), from the captured dL/dh of the heads (top
    layer) or the captured d_gi(upper) . W_ih(upper) (lower layers).  The recurrent term d_gh . W_hh is taken from the product's
    own d_gh (rounded to bf16 with dgh_bf16) and W_hh (rounded to bf16 with whh='bf16'), so no error compounds through it."""
    B, T, H, top = c.B, c.T, c.H, c.top
    errs = {}
    g_top = {"f": c.g_hcat[:, :H], "s": c.g_hcat[:, H:2 * H], "b": c.g_hcat[:, 2 * H:]}
    for l in range(top, -1, -1):
        dy = {}
        if l < top:
            u = l + 1
            w = {d: c.params[pname(u, d, "weight_ih")].double() for d in ("f", "b", "s")}
            dy_f = c.dgi[(u, "f")].double() @ w["f"]
            dy_r = c.dgi[(u, "b")].double() @ w["b"]
            nr = c.dgi[(u, "s")].shape[0]
            dy_r[:nr] += c.dgi[(u, "s")].double() @ w["s"]
            dy = {"f": (dy_f, 0), "b": (dy_r, H), "s": (dy_r, 0)}
        for d in ("f", "b", "s"):
            j = (l, d)
            single = l == top and d == "s"
            w_hh = c.params[pname(l, d, "weight_hh")]
            w_hh = bf(w_hh) if whh == "bf16" else w_hh.double()
            gates, seq = c.layers[l]["gates"][d], c.layers[l]["seq"].get(d)
            g = g_top[d].double() if l == top else torch.zeros(B, H, device=DEV, dtype=torch.float64)
            for s in range(0 if single else T - 1, -1, -1):
                if dy:
                    src, c0 = dy[d]
                    r0 = t_out(l, d, s, top, T) * B
                    g = g + src[r0:r0 + B, c0:c0 + H]
                gt = gates[0 if single else t_out(l, d, s, top, T)].double()
                r, z, n, hn = gt[:, :H], gt[:, H:2 * H], gt[:, 2 * H:3 * H], gt[:, 3 * H:]
                hp = 0.0 if s == 0 else seq[s - 1].double()
                ga = g * (1 - z) * (1 - n * n)
                gz = g * (hp - n) * z * (1 - z)
                gr = ga * hn * r * (1 - r)
                ref_gi, ref_gh = torch.cat([gr, gz, ga], 1), torch.cat([gr, gz, ga * r], 1)
                ti = 0 if single else t_in(l, d, s, top, T)
                got_gi, got_gh = c.dgi[j][ti * B:(ti + 1) * B], c.dgh[j][s * B:(s + 1) * B]
                errs[(l, d, s)] = (rel(got_gi, ref_gi), rel(got_gh, ref_gh))
                g = g * z
                if s > 0:
                    g = g + (bf(got_gh) if dgh_bf16 else got_gh.double()) @ w_hh
    return errs


# ------------------------------------------------------------------------------------------------------------- stages
CASES = [pytest.param(*shape, tc, id=f"{sid}-{'tc' if tc else 'ffma'}") for shape, sid in zip(SHAPES, SHAPE_IDS) for tc in (False, True)]


@pytest.mark.parametrize("seed,L,H,B,T,tc", CASES)
def test_forward_gates_and_states_match_float64_cell(seed, L, H, B, T, tc):
    """Every step of every job of every layer (the top layer's single-step "s" job included): the saved r, z, n and h_t within
    FWD_ABS = 4e-5 absolute, gh_n within FWD_GHN = 1e-5 of max |gh_n|, of a float64 cell on the product's own bf16-rounded
    operands; NaN-filled buffers, so a skipped gate store fails.  Control: the same cell on unrounded operands misses FWD_ABS.
    Measured on a B200: r, z, n, h 9.5e-6, gh_n 1.5e-6; control 7.0e-3 at least."""
    c = step(seed, L, H, B, T, tc)
    worst = forward_errors(c)
    print("forward worst per job: " + ", ".join(f"{j}: " + " ".join(f"{k}={v:.1e}" for k, v in e.items()) for j, e in worst.items()))
    bad = {j: e for j, e in worst.items() if not (max(e["r"], e["z"], e["n"], e["h"]) <= FWD_ABS and e["gh_n"] <= FWD_GHN)}
    assert not bad, bad
    # the top layer's final states are the ones the heads read
    seq = c.layers[c.top]["seq"]
    assert torch.equal(c.h_cat[:, :H], seq["f"][T - 1]) and torch.equal(c.h_cat[:, 2 * H:], seq["b"][T - 1])
    ctrl = max(max(e["r"], e["z"], e["n"], e["h"]) for e in forward_errors(c, rnd=lambda t: t.double()).values())
    print(f"forward control (unrounded operands) {ctrl:.2e}")
    assert ctrl > FWD_ABS, ctrl


@pytest.mark.parametrize("seed,L,H,B,T,tc", CASES)
def test_bptt_matches_float64_adjoint_on_own_operands(seed, L, H, B, T, tc):
    """Every job and step: d_gi and d_gh within BPTT_REL = 1e-5 (max-norm relative) of the float64 replay with bf16(W_hh) and the
    product's bf16-rounded d_gh in the recurrent term.  Control: with fp32 W_hh in that term the replay misses the same bar at
    some step (wherever there is a recurrent term, T > 1).  Measured on a B200: worst 1.0e-6; control 4.8e-4 at least."""
    c = step(seed, L, H, B, T, tc)
    errs = bptt_errors(c)
    worst = max(max(v) for v in errs.values())
    print(f"bptt worst {worst:.2e} over {len(errs)} job-steps")
    bad = {k: v for k, v in errs.items() if not max(v) <= BPTT_REL}
    assert not bad, bad
    assert len(errs) == 3 * T * c.top + 2 * T + 1
    if T > 1:
        ctrl = max(max(v) for v in bptt_errors(c, whh="fp32").values())
        print(f"bptt control (fp32 W_hh in the reference) {ctrl:.2e}")
        assert ctrl > BPTT_REL, ctrl


@pytest.mark.parametrize("seed,L,H,B,T", [pytest.param(*s, id=i) for s, i in zip(SHAPES, SHAPE_IDS) if s[4] > 1 and s[2] >= 256])
def test_fp32_bptt_branch_matches_float64_adjoint(seed, L, H, B, T):
    """train_fp32_bptt=True on a bf16 model: the recurrent term runs on the fp32 GEMM over fp32 W_hh; the replay takes fp32
    d_gh and W_hh.  Same bar, BPTT_REL = 1e-5.  Measured on a B200: worst 8.1e-7."""
    c = step(seed, L, H, B, T, True, fp32_bptt=True)
    errs = bptt_errors(c, whh="fp32", dgh_bf16=False)
    worst = max(max(v) for v in errs.values())
    print(f"fp32 bptt worst {worst:.2e}")
    bad = {k: v for k, v in errs.items() if not max(v) <= BPTT_REL}
    assert not bad, bad


@pytest.mark.parametrize("seed,L,H,B,T,tc", CASES)
def test_gradients_match_float64_on_own_operands(seed, L, H, B, T, tc):
    """Every weight-gradient GEMM of the step passes gemm_check (ratio <= 1, no NaN) on its exact operands: bf16(g^T), bf16(x^T)
    when it ran on the tensor cores, fp32 otherwise.  Control: on the unrounded operands every tensor-core call exceeds the
    bound.  Every bias gradient (a column sum of the captured d_gi / d_gh, or of the regressor's and heads' adjoints) passes
    the same bound against the float64 sum.  The heads' weight gradients pass it on their own operands, g_feat^T relu(h): the
    bf16 forward flips a few relu masks, which moved them 1.06e-2 from the fp32 oracle at B = 3, T = 1.  The regressor
    gradients stay within REGRESSOR_REL = 1e-2 of the fp32 oracle.  Measured on a B200: worst ratio 0.38; smallest control
    ratio 62; regressor 3.4e-3."""
    c = step(seed, L, H, B, T, tc)
    ratios, controls = {}, {}
    for rec, name in zip(c.wg, c.wg_names):
        g, x, out = rec["g"], rec["x"], rec["out"]
        on_tc = rec["tensor_core"] and out.shape[0] % 16 == 0
        a, w = (g.T.to(torch.bfloat16), x.T.to(torch.bfloat16)) if on_tc else (g.T, x.T)
        chk = gemm_check(a, w, None, None, False, out)
        assert chk.nans == 0, (name, chk)
        ratios[name] = chk.ratio
        if on_tc:
            controls[name] = gemm_check(g.T, x.T, None, None, False, out).ratio
    g2 = c.g_feat.reshape(B, 2, 2048)
    for name, g_rows, lo, hi in (("encoder.linear_fwd.weight", g2[:, 0], 0, H), ("encoder.linear_rec.weight", g2[:, 1], H, 3 * H)):
        chk = gemm_check(g_rows.T, c.h_cat[:, lo:hi].clamp(min=0.0).T, None, None, False, c.grads[name])
        assert chk.nans == 0, (name, chk)
        ratios[name] = chk.ratio
    for rec, name in zip(c.cs, c.cs_names):
        a = rec["a"]
        chk = gemm_check(torch.ones(1, a.shape[0], device=DEV), a.T, None, None, False, rec["out"][None])
        assert chk.nans == 0, (name, chk)
        ratios["colsum " + name] = chk.ratio
        if name in c.grads:
            assert torch.equal(c.grads[name], rec["out"]), name
    print("worst gemm_check ratios: " + ", ".join(f"{k}={v:.2f}" for k, v in sorted(ratios.items(), key=lambda kv: -kv[1])[:4]))
    bad = {k: v for k, v in ratios.items() if not v <= 1.0}
    assert not bad, bad
    if tc:
        assert controls and len(controls) == sum(".gru_" in n for n in c.wg_names), controls
        print(f"smallest control ratio {min(controls.values()):.2f}")
        weak = {k: v for k, v in controls.items() if not v > 1.0}
        assert not weak, weak
    # the top layer's gru_rec forward direction is one step from h_0 = 0
    assert float(c.grads[f"encoder.gru_rec.weight_hh_l{c.top}"].abs().max()) == 0.0
    ref = oracle_grads(c)
    reg = {k: rel(c.grads[k].cpu(), v.double()) for k, v in ref.items() if k.startswith("regressor.")}
    assert len(reg) == 10
    print(f"regressor worst {max(reg.values()):.1e}")
    bad = {k: v for k, v in reg.items() if not v < REGRESSOR_REL}
    assert not bad, bad


# ------------------------------------------------------------------------------------------------------------- launchers
def _nan(*shape, dtype=torch.float32):
    return torch.full(shape, float("nan"), device=DEV, dtype=dtype)


def _rand(rows, cols, ld, seed):
    """[rows, ld] fp32 buffer whose [rows, cols] window is random and whose padding columns are NaN."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    buf = _nan(max(rows, 1), ld)
    buf[:rows, :cols] = torch.randn(rows, cols, device=DEV, generator=g)
    return buf


# (rows, cols, ld) with rows / cols off multiples of 32, ld > cols, zero rows
RAGGED = [(0, 7, 9), (1, 33, 40), (37, 45, 45), (45, 100, 103), (257, 65, 70), (1000, 31, 33)]


@pytest.mark.parametrize("bf16", [False, True])
@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("rows,cols,ld_src,ld_dst,dst_rows", [(0, 7, 9, 4, 8), (1, 33, 40, 64, 33), (37, 45, 45, 40, 64),
                                                              (70, 3, 3, 72, 16), (100, 130, 131, 128, 130), (257, 65, 70, 260, 65)])
def test_transpose_launcher(rows, cols, ld_src, ld_dst, dst_rows, relu, bf16):
    """dst [dst_rows, ld_dst] = the transposed (optionally relu'd, bf16-rounded) window, zero elsewhere; the buffer is NaN-filled
    and followed by a NaN guard that must survive."""
    src = _rand(rows, cols, ld_src, rows * 7 + cols)
    dt = torch.bfloat16 if bf16 else torch.float32
    buf = _nan(dst_rows * ld_dst + 64, dtype=dt)
    nv.check(nv.lib().tp_transpose_f32(nv.ptr(src), ld_src, rows, cols, nv.ptr(buf), ld_dst, dst_rows,
                                       nv.PRECISION_BF16 if bf16 else nv.PRECISION_FP32, 1 if relu else 0, nv.stream()))
    torch.cuda.synchronize()
    want = torch.zeros(dst_rows, ld_dst, device=DEV, dtype=torch.float64)
    v = src[:rows, :cols].double()
    want[:cols, :rows] = (v.clamp(min=0.0) if relu else v).T
    got = buf[:dst_rows * ld_dst].view(dst_rows, ld_dst).double()
    assert torch.equal(got, want.to(dt).double())
    assert torch.isnan(buf[dst_rows * ld_dst:].float()).all()


@pytest.mark.parametrize("beta", [0.0, 0.75])
@pytest.mark.parametrize("rows,cols,ld", RAGGED)
def test_colsum_launcher(rows, cols, ld, beta):
    """out = beta out + column sums, within the gemm_check bound of the float64 sum; with beta = 0 a NaN-filled out is overwritten."""
    a = _rand(rows, cols, ld, rows + 3 * cols)
    out = _nan(cols + 16)
    if beta:
        out[:cols] = torch.randn(cols, device=DEV)
    before = out[:cols].double()
    nv.check(nv.lib().tp_colsum_f32(nv.ptr(a), ld, rows, cols, nv.ptr(out), beta, nv.stream()))
    torch.cuda.synchronize()
    # [beta | 1 ... 1] . [out_before | A]^T: the same accumulation bound as a GEMM over rows + 1 terms
    ones = torch.cat([torch.full((1,), beta, device=DEV, dtype=torch.float64), torch.ones(rows, device=DEV, dtype=torch.float64)])
    opnd = torch.cat([(before if beta else torch.zeros_like(before))[:, None], a[:rows, :cols].double().T], 1)
    chk = gemm_check(ones[None], opnd, None, None, False, out[None, :cols])
    assert chk.nans == 0 and chk.ratio <= 1.0, chk
    assert torch.isnan(out[cols:]).all()


@pytest.mark.parametrize("alpha,beta", [(1.0, 0.0), (1.0, 1.0), (-0.5, 0.25)])
@pytest.mark.parametrize("rows,cols,ld", RAGGED)
def test_axpby_launcher(rows, cols, ld, alpha, beta):
    src = _rand(rows, cols, ld, rows + cols)
    dst = _rand(rows, cols, ld + 5, 2 * rows + cols)
    if beta == 0.0:
        dst[:rows, :cols] = float("nan")            # beta = 0 overwrites, whatever dst held
    s = alpha * src[:rows, :cols].double()
    d0 = beta * dst[:rows, :cols].double() if beta else torch.zeros_like(s)
    pad = dst[:, cols:].clone()
    nv.check(nv.lib().tp_axpby_f32(nv.ptr(src), ld, nv.ptr(dst), ld + 5, rows, cols, alpha, beta, nv.stream()))
    torch.cuda.synchronize()
    err = (dst[:rows, :cols].double() - (s + d0)).abs()
    assert not torch.isnan(err).any() and bool((err <= 3 * 2.0 ** -24 * (s.abs() + d0.abs())).all())
    assert torch.isnan(dst[:, cols:]).all() and torch.isnan(pad).all()


@pytest.mark.parametrize("rows,cols,ld", RAGGED)
def test_mask_scale_and_relu_backward_launchers(rows, cols, ld):
    """a *= mask * scale and g = (h > 0) ? g : 0 inside the window only (NaN padding of a, g untouched; NaN padding of mask, h
    never read)."""
    g0 = torch.Generator(device=DEV).manual_seed(rows + cols)
    mask = _nan(max(rows, 1), ld + 3)
    mask[:rows, :cols] = (torch.rand(rows, cols, device=DEV, generator=g0) >= 0.5).float()
    a = _rand(rows, cols, ld, rows)
    want = a[:rows, :cols].double() * mask[:rows, :cols].double() * 2.0
    nv.check(nv.lib().tp_mask_scale(nv.ptr(a), ld, nv.ptr(mask), ld + 3, rows, cols, 2.0, nv.stream()))
    h = _rand(rows, cols, ld + 1, cols)
    h[:rows, :cols][h[:rows, :cols].abs() < 0.3] = 0.0          # exact zeros: relu'(0) = 0, as torch.relu's backward
    g = _rand(rows, cols, ld, 5 * rows)
    want_g = torch.where(h[:rows, :cols] > 0, g[:rows, :cols], torch.zeros_like(g[:rows, :cols])).double()
    nv.check(nv.lib().tp_relu_backward(nv.ptr(g), ld, nv.ptr(h), ld + 1, rows, cols, nv.stream()))
    torch.cuda.synchronize()
    assert torch.equal(a[:rows, :cols].double(), want)          # mask in {0, 1}, scale 2: exact
    assert torch.equal(g[:rows, :cols].double(), want_g)
    assert torch.isnan(a[:, cols:]).all() and torch.isnan(g[:, cols:]).all()


@pytest.mark.parametrize("k_in", [16, 157, 2176])
@pytest.mark.parametrize("n_out", [16, 48, 6144])
@pytest.mark.parametrize("rows", [1, 20, 63, 64, 65, 480])
def test_tensor_core_weight_grad_sweep(monkeypatch, rows, n_out, k_in):
    """_Ops.weight_grad(tensor_core=True) against float64 on bf16(g^T), bf16(x^T) (gemm_check), over reductions that are not,
    are, and just pass a multiple of the 64-row padding, and k_in % 16 != 0 (the scratch-and-copy branch).  Inputs carry NaN
    past the rows and columns the GEMM reads, and out and every torch.empty of train.py are NaN-filled."""
    monkeypatch.setattr(tr, "torch", _NaNTorch())
    gen = torch.Generator(device=DEV).manual_seed(rows * 131 + n_out + k_in)
    g = _nan(rows + 3, n_out)
    g[:rows] = torch.randn(rows, n_out, device=DEV, generator=gen)
    x = _nan(rows + 3, k_in + 5)
    x[:rows, :k_in] = torch.randn(rows, k_in, device=DEV, generator=gen)
    out = _nan(n_out, k_in)
    tr._Ops.weight_grad(g, x[:, :k_in], out, rows, tensor_core=True)
    torch.cuda.synchronize()
    chk = gemm_check(g[:rows].T.to(torch.bfloat16), x[:rows, :k_in].T.to(torch.bfloat16), None, None, False, out)
    assert chk.nans == 0 and chk.ratio <= 1.0, chk
    ctrl = gemm_check(g[:rows].T, x[:rows, :k_in].T, None, None, False, out)
    assert ctrl.ratio > 1.0, ctrl              # the bf16 rounding is visible at this bound


# ------------------------------------------------------------------------------------------------------------- fp32_tc
@pytest.mark.parametrize("seed,B,T,H", [(86, 4, 6, 256), (0, 32, 16, 2048)], ids=["small", "configs4"])
def test_fp32_tc_train_step_meets_fp32_bar(seed, B, T, H):
    """precision='fp32_tc' in train mode (split-bf16 K1 / K2 with the gates saved by the BF16X3 recurrence, then the fp32
    backward): loss within 1e-4 relative and every parameter gradient within 1e-4 max-norm relative of torch.autograd
    through the oracle, the bar of the fp32 step.  Measured on a B200: worst 2.4e-5 (small), 1.0e-5 (configs[4])."""
    model, sd = build_product_model(seed, T, 1, H, "fp32_tc", DEV)
    model.train()
    x = synth.make_input(seed, B, T)
    masks = train_ref.make_masks(seed, 2 * B)
    tgt = train_ref.make_targets(seed, 2 * B)
    out = model(torch.from_numpy(x).to(DEV), is_train=True, dropout_masks=torch.from_numpy(masks).to(DEV))[-1]
    loss = train_ref.synthetic_loss(out, tgt)
    loss.backward()
    _, ref_loss, ref_grads = train_ref.TrainOracle(sd, seed, 1, H).loss_and_grads(x, masks, tgt)
    assert abs(float(loss.detach()) - ref_loss) < 1e-4 * max(1.0, abs(ref_loss))
    params = dict(model.named_parameters())
    worst = {name: rel(params[name].grad.cpu(), g_ref.double()) for name, g_ref in ref_grads.items()}
    print("fp32_tc worst gradient errors:", {k: f"{v:.1e}" for k, v in sorted(worst.items(), key=lambda kv: -kv[1])[:4]})
    bad = {k: v for k, v in worst.items() if not v < 1e-4}
    assert not bad, bad
