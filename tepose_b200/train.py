"""Training step of the path: train-mode forward (dropout masks as inputs), hand-written backward, data-parallel gradient
all-reduce (BASELINE.json configs[4]).

What the reference does (paths relative to the reference repository):
    lib/core/trainer.py:137,203      generator.train(); preds = generator(inp, is_train=True)
    lib/models/tepose.py:85,138-145  train mode regresses the fwd- and the rec-feature separately: outputs are [B, 2, ...]
    lib/models/spin.py:216-218,253-261  drop1 / drop2 (p = 0.5) are active inside the 3 IEF iterations
    lib/core/trainer.py:235-237      gen_optimizer.zero_grad(); loss.backward(); gen_optimizer.step()   (torch.autograd)
    lib/utils/utils.py:145-152       Adam over all parameters
Here `TePose.forward` in `.train()` mode routes through `TrainFunction` (a torch.autograd.Function): the forward runs the same
K1/K2 kernels with the per-step gate activations saved, the IEF as explicit GEMMs with `tp_mask_scale`, and the fused SMPL
kernels; the backward is csrc/train.cu (SMPL / rotation / GRU-cell adjoints) + the library GEMMs on transposed operands.
Dropout masks are INPUTS (SURVEY.md H8): `forward(..., dropout_masks=m)` with m [n_iter, 2, 2B, 1024] in {0,1}; when omitted
they are drawn with torch.rand on the device (what nn.Dropout does with its own generator).

Scope: any n_layers, including the released configuration (L = 2, H = 1024, T = 6) that every training config of the reference
sets.  The backward walks the encoder top-down with one back-propagation-through-time loop for every (layer, direction): below
the top layer, the gradient of a layer's output sequence is d_gi . W_ih of the layer above (one GEMM per upper direction) and
is added to dL/dh before each step's cell adjoint.  Gradients flow to every encoder / regressor parameter, not to the input
features.  `DataParallel` at the bottom is the one place of the package that uses a collective: one NCCL all-reduce
per gradient bucket, launched from inside the backward as soon as a bucket is complete so that it overlaps the BPTT.
"""
from __future__ import annotations

import torch

from . import _native as nv
from .spin import PSC

DROP_P = 0.5
N_ITER = 3


def _up(v, m):
    return (v + m - 1) // m * m


class _Ops:
    """Thin launch helpers over the C ABI (fp32 row-major tensors, last stride 1)."""

    @staticmethod
    def gemm(a, w, out=None, bias=None, cin=None, alpha=1.0, beta=0.0, M=None, N=None, K=None):
        """out[M,N] = alpha * (a[M,K] . w[N,K]^T + bias) + beta * cin   (tp_gemm_f32; split-K when the tile grid is small)."""
        L = nv.lib()
        M = a.shape[0] if M is None else M
        N = w.shape[0] if N is None else N
        K = a.shape[1] if K is None else K
        if out is None:
            out = torch.empty(M, N, device=a.device, dtype=torch.float32)
        P = lambda t: nv.vp(0) if t is None else nv.vp(t.data_ptr())
        bm, bn = (32, 32) if M <= 32 else ((64, 32) if M <= 64 else (128, 64))
        tiles = ((M + bm - 1) // bm) * ((N + bn - 1) // bn)
        splits = 1 if tiles >= 120 else max(1, min(K // 128, 240 // max(tiles, 1), 32))
        ldcin = 0 if cin is None else cin.stride(0)
        if splits > 1 and tiles <= 1024:
            ws = nv.workspace(int(L.tp_gemm_f32_splitk_workspace_bytes(M, N, splits)), a.device)
            ws[:4096].zero_()
            nv.check(L.tp_gemm_f32_splitk(P(a), a.stride(0), P(w), w.stride(0), P(bias), P(cin), ldcin, P(out), out.stride(0),
                                          M, N, K, alpha, beta, 0, splits, nv.ptr(ws), ws.numel(), nv.stream()), "tp_gemm_f32_splitk")
        else:
            nv.check(L.tp_gemm_f32(P(a), a.stride(0), P(w), w.stride(0), P(bias), P(cin), ldcin, P(out), out.stride(0),
                                   M, N, K, alpha, beta, 0, nv.stream()), "tp_gemm_f32")
        return out

    @staticmethod
    def transpose(src, rows=None, cols=None, relu=False, dst_rows=None, bf16=False):
        """[rows, cols] (row stride src.stride(0)) -> [dst_rows >= cols, ld] with ld = rows rounded up (zero padded)."""
        rows = src.shape[0] if rows is None else rows
        cols = src.shape[1] if cols is None else cols
        ld = _up(max(rows, 1), 64 if bf16 else 4)
        dst_rows = cols if dst_rows is None else dst_rows
        out = torch.empty(dst_rows, ld, device=src.device, dtype=torch.bfloat16 if bf16 else torch.float32)
        nv.check(nv.lib().tp_transpose_f32(nv.vp(src.data_ptr()), src.stride(0), rows, cols, nv.vp(out.data_ptr()), ld, dst_rows,
                                           nv.PRECISION_BF16 if bf16 else nv.PRECISION_FP32, 1 if relu else 0, nv.stream()), "tp_transpose_f32")
        return out

    @staticmethod
    def colsum(a, rows=None, cols=None):
        rows = a.shape[0] if rows is None else rows
        cols = a.shape[1] if cols is None else cols
        out = torch.empty(cols, device=a.device, dtype=torch.float32)
        nv.check(nv.lib().tp_colsum_f32(nv.vp(a.data_ptr()), a.stride(0), rows, cols, nv.ptr(out), 0.0, nv.stream()), "tp_colsum_f32")
        return out

    @staticmethod
    def mask_scale(a, mask, scale):
        nv.check(nv.lib().tp_mask_scale(nv.vp(a.data_ptr()), a.stride(0), nv.vp(mask.data_ptr()), mask.stride(0), a.shape[0], a.shape[1],
                                        scale, nv.stream()), "tp_mask_scale")

    @staticmethod
    def relu_backward(g, h):
        nv.check(nv.lib().tp_relu_backward(nv.vp(g.data_ptr()), g.stride(0), nv.vp(h.data_ptr()), h.stride(0), g.shape[0], g.shape[1],
                                           nv.stream()), "tp_relu_backward")

    @staticmethod
    def weight_grad(g, x, out, rows, tensor_core=False):
        """out[Nout, Kin] = g[rows, Nout]^T . x[rows, Kin]  (dW of y = x W^T): both operands are transposed so that the reduction
        dimension (the rows) is contiguous, then one library GEMM.  tensor_core: bf16 operands on the tcgen05 GEMM (fp32 out)."""
        n_out, k_in = out.shape
        if tensor_core and n_out % 16 == 0:
            gT = _Ops.transpose(g, rows, n_out, bf16=True)
            xT = _Ops.transpose(x, rows, k_in, dst_rows=_up(k_in, 16), bf16=True)
            seg = (nv.GemmSeg * 1)(nv.GemmSeg(0, n_out, 0, k_in if k_in % 16 == 0 else _up(k_in, 16), nv.ptr(out), out.stride(0), nv.vp(0)))
            if k_in % 16 == 0:
                nv.check(nv.lib().tp_gemm_bf16_tc(nv.ptr(gT), n_out, nv.ptr(xT), xT.shape[0], gT.shape[1], seg, 1, nv.stream()), "tp_gemm_bf16_tc")
                return out
            tmp = torch.empty(n_out, _up(k_in, 16), device=out.device, dtype=torch.float32)
            seg[0].out, seg[0].ldc = tmp.data_ptr(), tmp.stride(0)
            nv.check(nv.lib().tp_gemm_bf16_tc(nv.ptr(gT), n_out, nv.ptr(xT), xT.shape[0], gT.shape[1], seg, 1, nv.stream()), "tp_gemm_bf16_tc")
            out.copy_(tmp[:, :k_in])
            return out
        gT = _Ops.transpose(g, rows, n_out)
        xT = _Ops.transpose(x, rows, k_in)
        return _Ops.gemm(gT, xT, out=out, M=n_out, N=k_in, K=gT.shape[1])


class TrainFunction(torch.autograd.Function):
    """(theta, verts, kp_2d, kp_3d, rotmat) = f(x, masks; parameters) with a hand-written backward."""

    @staticmethod
    def forward(ctx, model, x, masks, *params):
        outs, saved = _train_forward(model, x, masks)
        ctx.model, ctx.saved = model, saved
        ctx.set_materialize_grads(False)        # outputs the loss does not use (verts, rotmat) arrive as None, not as zeros
        return outs

    @staticmethod
    def backward(ctx, g_theta, g_verts, g_kp2d, g_kp3d, g_rotmat):
        grads = _train_backward(ctx.model, ctx.saved, g_theta, g_verts, g_kp2d, g_kp3d, g_rotmat)
        ctx.saved = None
        return (None, None, None) + tuple(grads)


def path_parameters(model):
    """The parameters the path reads, in a fixed order (regressor.smpl.* Parameters exist for state_dict parity only):
    the twelve GRU tensors of every layer, the linear heads, the regressor."""
    enc, reg = model.encoder, model.regressor
    kinds = ("weight_ih", "weight_hh", "bias_ih", "bias_hh")
    names = [f"gru_fwd.{k}_l{l}" for l in range(enc.n_layers) for k in kinds]
    names += [f"gru_rec.{k}_l{l}{sfx}" for l in range(enc.n_layers) for sfx in ("", "_reverse") for k in kinds]
    out = []
    for n in names:
        mod, attr = n.split(".")
        out.append(("encoder." + n, getattr(getattr(enc, mod), attr)))
    for mod in ("linear_fwd", "linear_rec"):
        out.append((f"encoder.{mod}.weight", getattr(enc, mod).weight))
        out.append((f"encoder.{mod}.bias", getattr(enc, mod).bias))
    for mod in ("fc1", "fc2", "decpose", "decshape", "deccam"):
        out.append((f"regressor.{mod}.weight", getattr(reg, mod).weight))
        out.append((f"regressor.{mod}.bias", getattr(reg, mod).bias))
    return out


def make_dropout_masks(n_rows, device, n_iter=N_ITER, generator=None):
    """Keep masks [n_iter, 2, n_rows, 1024] in {0,1} (Bernoulli(1 - p)), drawn on the device."""
    return (torch.rand(n_iter, 2, n_rows, 1024, device=device, generator=generator) >= DROP_P).float()


def train_forward(model, x, dropout_masks=None):
    """lib/models/tepose.py:121-147 with is_train=True under .train(): list of one dict with [B, 2, ...] outputs attached to the
    autograd graph of the model's parameters."""
    nv.require_cuda(x, "input")
    B = x.shape[0]
    if dropout_masks is None:
        dropout_masks = make_dropout_masks(2 * B, x.device)
    if tuple(dropout_masks.shape[1:]) != (2, 2 * B, 1024):
        raise ValueError(f"dropout_masks must be [n_iter, 2, {2 * B}, 1024], got {tuple(dropout_masks.shape)}")
    params = [p for _, p in path_parameters(model)]
    theta, verts, kp2d, kp3d, rotmat = TrainFunction.apply(model, x, dropout_masks.float().contiguous(), *params)
    return [{"theta": theta.reshape(B, 2, -1), "verts": verts.reshape(B, 2, -1, 3), "kp_2d": kp2d.reshape(B, 2, -1, 2),
             "kp_3d": kp3d.reshape(B, 2, -1, 3), "rotmat": rotmat.reshape(B, 2, -1, 3, 3)}]


# ------------------------------------------------------------------------------------------------------------ forward
def _train_forward(model, x, masks):
    enc, reg = model.encoder, model.regressor
    dev, H = x.device, enc.hidden_size
    B, T = x.shape[0], x.shape[1]
    N = 2 * B
    with torch.cuda.device(dev):
        sv = {"B": B, "T": T, "masks": masks}
        # K1 + K2 with every step's state and gate activations kept
        h_fwd, h_rec = enc.encode_states(x, train_ctx=sv)
        h_cat = torch.as_strided(h_fwd, (B, 3 * H), (3 * H, 1))
        sv["h_cat"] = h_cat
        feat = enc.heads(h_fwd, h_rec, is_train=True).reshape(N, 2048)           # rows (b, 0) = fwd, (b, 1) = rec
        sv["feat"] = feat
        # IEF with dropout (lib/models/spin.py:250-261): fc1 is split into its feature part (iteration invariant) and its
        # [pose|shape|cam] part; decpose / decshape / deccam are one stacked [160,1024] matrix (Regressor.packed(), fp32)
        pk = reg.packed() if reg.precision == "fp32" else _fp32_regressor_pack(reg)
        scale = 1.0 / (1.0 - DROP_P)
        n_iter = masks.shape[0]
        psc_all = torch.empty(n_iter + 1, N, PSC, device=dev, dtype=torch.float32)
        psc_all[0] = pk["init"]
        d1_all = torch.empty(n_iter, N, 1024, device=dev, dtype=torch.float32)
        d2_all = torch.empty(n_iter, N, 1024, device=dev, dtype=torch.float32)
        base1 = _Ops.gemm(feat, pk["w1x"], bias=pk["b1"])
        for i in range(n_iter):
            _Ops.gemm(psc_all[i], pk["w1p"], out=d1_all[i], cin=base1, beta=1.0)
            _Ops.mask_scale(d1_all[i], masks[i, 0], scale)
            _Ops.gemm(d1_all[i], pk["w2"], out=d2_all[i], bias=pk["b2"])
            _Ops.mask_scale(d2_all[i], masks[i, 1], scale)
            _Ops.gemm(d2_all[i], pk["wdec"], out=psc_all[i + 1], bias=pk["bdec"], cin=psc_all[i], beta=1.0)
        sv.update(psc_all=psc_all, d1_all=d1_all, d2_all=d2_all, reg_pack=pk)
        out = reg.decode(psc_all[n_iter], is_train=True)[0]
        sv["joints"], sv["rotmat"] = out["kp_3d"], out["rotmat"]
    return (out["theta"], out["verts"], out["kp_2d"], out["kp_3d"], out["rotmat"]), sv


def _fp32_regressor_pack(reg):
    """fp32 operand copies of the Regressor weights for the train path of a bf16-mode model (same layout as packed())."""
    saved = reg.precision
    reg.precision = "fp32"
    try:
        pk = dict(reg.packed())
    finally:
        reg.precision = saved
        reg._pack = None
    return pk


# ------------------------------------------------------------------------------------------------------------ backward
def _train_backward(model, sv, g_theta, g_verts, g_kp2d, g_kp3d, g_rotmat):
    enc, reg = model.encoder, model.regressor
    smpl = reg.smpl
    L = nv.lib()
    B, T, H = sv["B"], sv["T"], enc.hidden_size
    N = 2 * B
    psc_all, d1_all, d2_all, masks, pk = sv["psc_all"], sv["d1_all"], sv["d2_all"], sv["masks"], sv["reg_pack"]
    n_iter = masks.shape[0]
    dev = psc_all.device
    tc = bool(getattr(model, "train_tensor_core_grads", False))
    sync = getattr(model, "_grad_sync", None)
    P = lambda t: nv.vp(0) if t is None else nv.vp(t.data_ptr())
    cont = lambda t: None if t is None else t.detach().float().contiguous()
    with torch.cuda.device(dev):
        g_theta, g_verts, g_kp2d, g_kp3d, g_rotmat = (cont(t) for t in (g_theta, g_verts, g_kp2d, g_kp3d, g_rotmat))
        psc = psc_all[n_iter]
        R = sv["rotmat"].reshape(N * 24, 9)
        # ---- theta = [cam | axis-angle(R) | shape]  (spin.py:282-285) and the rotmat output itself
        g_R_extra = None if g_rotmat is None else g_rotmat.reshape(N * 24, 9).clone()
        if g_theta is not None:
            if g_R_extra is None:
                g_R_extra = torch.empty(N * 24, 9, device=dev, dtype=torch.float32)
                acc = 0
            else:
                acc = 1
            nv.check(L.tp_rotmat_to_angle_axis_backward(P(R), nv.vp(g_theta.data_ptr() + 12), 85, 24, P(g_R_extra), N * 24, acc, nv.stream()),
                     "tp_rotmat_to_angle_axis_backward")
        # ---- SMPL + projection adjoint
        p = smpl.packed()
        g_R = torch.empty(N * 24, 9, device=dev, dtype=torch.float32)
        g_betas = torch.empty(N, 10, device=dev, dtype=torch.float32)
        g_cam = torch.empty(N, 3, device=dev, dtype=torch.float32)
        ws = nv.workspace(L.tp_smpl_backward_workspace_bytes(p.c_model, N), dev)
        nv.check(L.tp_smpl_backward(p.c_model, N, P(R), nv.vp(psc.data_ptr() + 4 * 144), PSC, nv.vp(psc.data_ptr() + 4 * 154), PSC,
                                    P(smpl._jreg_extra), smpl._jreg_extra.shape[0], P(smpl._src49), 49, P(sv["joints"]),
                                    P(g_verts), P(g_kp3d), P(g_kp2d), P(g_R_extra), P(g_R), P(g_betas), P(g_cam), nv.ptr(ws), ws.numel(),
                                    nv.stream()), "tp_smpl_backward")
        g_psc = torch.zeros(N, PSC, device=dev, dtype=torch.float32)
        x6 = psc[:, :144].contiguous()
        g_x6 = torch.empty(N, 144, device=dev, dtype=torch.float32)
        nv.check(L.tp_rot6d_backward(P(x6), P(g_R), P(g_x6), N * 24, nv.stream()), "tp_rot6d_backward")
        g_psc[:, :144] = g_x6
        g_psc[:, 144:154] = g_betas
        g_psc[:, 154:157] = g_cam
        if g_theta is not None:
            g_psc[:, 144:154] += g_theta[:, 75:85]
            g_psc[:, 154:157] += g_theta[:, 0:3]
        # ---- IEF adjoint (3 iterations, reversed)
        w1pT, w2T, wdecT = _Ops.transpose(pk["w1p"]), _Ops.transpose(pk["w2"]), _Ops.transpose(pk["wdec"])
        ga1_all = torch.empty(n_iter, N, 1024, device=dev, dtype=torch.float32)
        ga2_all = torch.empty(n_iter, N, 1024, device=dev, dtype=torch.float32)
        gdec_all = torch.empty(n_iter, N, PSC, device=dev, dtype=torch.float32)
        scale = 1.0 / (1.0 - DROP_P)
        for i in range(n_iter - 1, -1, -1):
            gdec_all[i].copy_(g_psc)
            _Ops.gemm(g_psc, wdecT, out=ga2_all[i])                                   # dL/d(drop2 output) = g_dec . Wdec
            _Ops.mask_scale(ga2_all[i], masks[i, 1], scale)
            _Ops.gemm(ga2_all[i], w2T, out=ga1_all[i])
            _Ops.mask_scale(ga1_all[i], masks[i, 0], scale)
            _Ops.gemm(ga1_all[i], w1pT, out=g_psc, cin=g_psc, beta=1.0)               # residual + fc1's state columns
        ga1_sum = ga1_all.sum(dim=0)
        g_feat = _Ops.gemm(ga1_sum, _Ops.transpose(pk["w1x"]))                        # [N, 2048]
        grads = {}
        fc1_g = torch.empty(1024, 2205, device=dev, dtype=torch.float32)
        dw1x = torch.empty(1024, 2048, device=dev, dtype=torch.float32)
        _Ops.weight_grad(ga1_sum, sv["feat"], dw1x, N)
        dw1p = torch.empty(1024, PSC, device=dev, dtype=torch.float32)
        _Ops.weight_grad(ga1_all.reshape(n_iter * N, 1024), psc_all[:n_iter].reshape(n_iter * N, PSC), dw1p, n_iter * N)
        fc1_g[:, :2048] = dw1x
        fc1_g[:, 2048:] = dw1p[:, :157]
        grads["regressor.fc1.weight"] = fc1_g
        grads["regressor.fc1.bias"] = _Ops.colsum(ga1_all.reshape(n_iter * N, 1024))
        dw2 = torch.empty(1024, 1024, device=dev, dtype=torch.float32)
        _Ops.weight_grad(ga2_all.reshape(n_iter * N, 1024), d1_all.reshape(n_iter * N, 1024), dw2, n_iter * N)
        grads["regressor.fc2.weight"] = dw2
        grads["regressor.fc2.bias"] = _Ops.colsum(ga2_all.reshape(n_iter * N, 1024))
        dwdec = torch.empty(PSC, 1024, device=dev, dtype=torch.float32)
        _Ops.weight_grad(gdec_all.reshape(n_iter * N, PSC), d2_all.reshape(n_iter * N, 1024), dwdec, n_iter * N)
        dbdec = _Ops.colsum(gdec_all.reshape(n_iter * N, PSC))
        for name, lo, hi in (("decpose", 0, 144), ("decshape", 144, 154), ("deccam", 154, 157)):
            grads[f"regressor.{name}.weight"] = dwdec[lo:hi].contiguous()
            grads[f"regressor.{name}.bias"] = dbdec[lo:hi].contiguous()
        # ---- linear heads + relu (tepose.py:79-85; rows (b,0) -> linear_fwd, (b,1) -> linear_rec)
        g2 = g_feat.reshape(B, 2, 2048)
        g_f, g_r = g2[:, 0], g2[:, 1]                                                  # row stride 4096
        f32 = lambda t: t.detach().float().contiguous()
        h_cat = sv["h_cat"]
        g_hcat = torch.empty(B, 3 * H, device=dev, dtype=torch.float32)
        _Ops.gemm(g_f, _Ops.transpose(f32(enc.linear_fwd.weight)), out=g_hcat[:, :H])
        _Ops.gemm(g_r, _Ops.transpose(f32(enc.linear_rec.weight)), out=g_hcat[:, H:])
        _Ops.relu_backward(g_hcat, h_cat)
        layers = sv["layers"]
        Ln = len(layers)
        top = Ln - 1
        dbg = getattr(model, "_debug_capture", None)
        if dbg is not None:
            dbg.update(g_hcat=g_hcat.clone(), h_cat=h_cat.clone(), g_feat=g_feat.clone(), seq_f=layers[top]["seq"]["f"].clone(),
                       seq_b=layers[top]["seq"]["b"].clone(), gates_f=layers[top]["gates"]["f"].clone(),
                       gates_b=layers[top]["gates"]["b"].clone())
        for name, g_rows, lo, hi in (("linear_fwd", g_f, 0, H), ("linear_rec", g_r, H, 3 * H)):
            dw = torch.empty(2048, hi - lo, device=dev, dtype=torch.float32)
            gT = _Ops.transpose(g_rows, B, 2048)
            hT = _Ops.transpose(h_cat[:, lo:hi], B, hi - lo, relu=True)
            _Ops.gemm(gT, hT, out=dw, M=2048, N=hi - lo, K=gT.shape[1])
            grads[f"encoder.{name}.weight"] = dw
            grads[f"encoder.{name}.bias"] = _Ops.colsum(g_rows, B, 2048)
        if sync is not None:
            sync.ready([(k, grads[k]) for k in grads])                                 # regressor + heads: first bucket, overlaps the BPTT
        # ---- GRU back-propagation through time, top layer first, over jobs (layer l, direction d): "f" = gru_fwd, "b" = the
        #      reverse direction of gru_rec, "s" = the forward direction of gru_rec.  In the top layer only the final states
        #      are consumed (SURVEY.md F3), and "s" is the single step at x_rec index 0 from h_0 = 0; below it every
        #      direction is full and takes the gradient of its whole output sequence from the layer above.
        def pname(l, d, k):
            return f"encoder.gru_fwd.{k}_l{l}" if d == "f" else f"encoder.gru_rec.{k}_l{l}" + ("_reverse" if d == "b" else "")

        def full(l):
            return ("f", "b") if l == top else ("f", "b", "s")

        def t_in(l, d, s):
            """Row block of the layer's input that step s reads: layer 0 reads x in original frame order, deeper layers of
            gru_rec read the x_rec-indexed sequence y_r (tau = T-1-t) of the layer below."""
            if d == "f":
                return s
            if d == "b":
                return s if l == 0 else T - 1 - s
            if l == top:
                return T - 1 if l == 0 else 0
            return T - 1 - s if l == 0 else s

        def t_out(l, d, s):
            """Row block that step s writes of the output sequence (and of the saved gates)."""
            return T - 1 - s if d == "b" and l != top else s

        param = dict(model.named_parameters())
        seq = {(l, d): layers[l]["seq"][d] for l in range(Ln) for d in full(l)}
        gates = {(l, d): layers[l]["gates"][d] for l in range(Ln) for d in ("f", "b", "s")}
        g_h = {(top, "f"): g_hcat[:, :H].contiguous(), (top, "s"): g_hcat[:, H:2 * H].contiguous(), (top, "b"): g_hcat[:, 2 * H:].contiguous()}
        whhT = {(l, d): _Ops.transpose(f32(param[pname(l, d, "weight_hh")])) for l in range(top, -1, -1) for d in full(l)}
        # mixed precision (precision='bf16' models): the per-step dL/dh += d_gh . W_hh runs on the skinny tensor-core GEMM over a
        # fragment-packed bf16 copy of W_hh^T (25 MB streamed per step instead of 50 MB of fp32 through the FFMA GEMM)
        whh_lp = None
        if model.precision == "bf16" and B <= 64 and H % 16 == 0 and not getattr(model, "train_fp32_bptt", False):
            whh_lp = {j: nv.pack_linear(w[:, :3 * H], "bf16") for j, w in whhT.items()}
            sk_splits = 8                                  # 128-row groups x 8 K slices: 128 CTAs stream W_hh^T at H = 2048
            sk_ws = nv.workspace(int(L.tp_skinny_bf16_workspace_bytes(B, H, sk_splits)), dev)
            sk_ws[:4096].zero_()
        # d_gi rows follow the layer's input (t_in), d_gh rows the run order (s)
        dgi = {j: torch.empty(T * B, 3 * H, device=dev, dtype=torch.float32) for j in whhT}
        dgh = {j: torch.empty(T * B, 3 * H, device=dev, dtype=torch.float32) for j in whhT}
        dgi[(top, "s")] = torch.empty(B, 3 * H, device=dev, dtype=torch.float32)
        dgh[(top, "s")] = torch.empty(B, 3 * H, device=dev, dtype=torch.float32)

        def cell(l, d, s):
            j = (l, d)
            single = j == (top, "s")
            ri = slice(0, B) if single else slice(t_in(l, d, s) * B, (t_in(l, d, s) + 1) * B)
            rh = slice(0, B) if single else slice(s * B, (s + 1) * B)
            hprev = seq[j][s - 1] if s > 0 else None
            nv.check(L.tp_gru_cell_backward(P(g_h[j]), H, nv.vp(gates[j].data_ptr() + 4 * t_out(l, d, s) * B * 4 * H), 4 * H,
                                            P(hprev), H, P(dgi[j][ri]), 3 * H, P(dgh[j][rh]), 3 * H, B, H, nv.stream()),
                     "tp_gru_cell_backward")

        for l in range(top, -1, -1):
            dy = {}
            if l < top:
                # layer boundary: dL/d(outputs of layer l) = d_gi of layer l+1 . W_ih of layer l+1, one GEMM per upper direction
                # over all T*B rows.  y_f [T*B, H] feeds "f" above; y_r [T*B, 2H] (columns [0,H) = this layer's "s",
                # [H,2H) = its "b", rows by tau) feeds "b" and "s" above -- the top layer's "s" reads only tau = 0.
                u = l + 1
                wT = {d: _Ops.transpose(f32(param[pname(u, d, "weight_ih")])) for d in ("f", "b", "s")}
                dy_f = _Ops.gemm(dgi[(u, "f")], wT["f"])
                dy_r = _Ops.gemm(dgi[(u, "b")], wT["b"])
                nr = dgi[(u, "s")].shape[0]
                _Ops.gemm(dgi[(u, "s")], wT["s"], out=dy_r[:nr], cin=dy_r[:nr], beta=1.0)
                dy = {"f": (dy_f, 0), "b": (dy_r, H), "s": (dy_r, 0)}
                for d in full(l):
                    g_h[(l, d)] = torch.empty(B, H, device=dev, dtype=torch.float32)
            else:
                cell(l, "s", 0)
            for s in range(T - 1, -1, -1):
                for d in full(l):
                    j = (l, d)
                    if dy:              # g_h += this step's output gradient (the first step of the walk starts from it)
                        src, c0 = dy[d]
                        r0 = t_out(l, d, s) * B
                        nv.check(L.tp_axpby_f32(nv.vp(src.data_ptr() + 4 * (r0 * src.stride(0) + c0)), src.stride(0), P(g_h[j]), H, B, H,
                                                1.0, 0.0 if s == T - 1 else 1.0, nv.stream()), "tp_axpby_f32")
                    cell(l, d, s)
                    if s > 0 and whh_lp is not None:
                        nv.check(L.tp_skinny_bf16(P(dgh[j][s * B:(s + 1) * B]), 3 * H, B, 3 * H, nv.ptr(whh_lp[j]), H, nv.vp(0), P(g_h[j]), H,
                                                  P(g_h[j]), H, 1.0, 1.0, 0, sk_splits, nv.ptr(sk_ws), sk_ws.numel(), nv.stream()), "tp_skinny_bf16")
                    elif s > 0:
                        _Ops.gemm(dgh[j][s * B:(s + 1) * B], whhT[j], out=g_h[j], cin=g_h[j], beta=1.0)
        if dbg is not None:
            dbg.update(dgi_f=dgi[(top, "f")].clone(), dgi_b=dgi[(top, "b")].clone(), dgh_f=dgh[(top, "f")].clone(),
                       dgh_b=dgh[(top, "b")].clone())
        # hidden-side weights: dW_hh = sum_t d_gh[t]^T h[t-1]  (rows B.. of d_gh against rows ..(T-1)B of the states)
        late = []
        for l in range(top, -1, -1):
            for d in full(l):
                j = (l, d)
                dw = torch.zeros(3 * H, H, device=dev, dtype=torch.float32)
                if T > 1:
                    _Ops.weight_grad(dgh[j][B:], seq[j].reshape(T * B, H), dw, (T - 1) * B, tensor_core=tc)
                grads[pname(l, d, "weight_hh")] = dw
                grads[pname(l, d, "bias_hh")] = _Ops.colsum(dgh[j])
                grads[pname(l, d, "bias_ih")] = _Ops.colsum(dgi[j])
                late += [pname(l, d, k) for k in ("weight_hh", "bias_hh", "bias_ih")]
            if l == top:
                j = (top, "s")
                grads[pname(top, "s", "weight_hh")] = torch.zeros(3 * H, H, device=dev, dtype=torch.float32)   # h_0 = 0: no gradient reaches it
                grads[pname(top, "s", "bias_hh")] = _Ops.colsum(dgh[j])
                grads[pname(top, "s", "bias_ih")] = _Ops.colsum(dgi[j])
                late += [pname(top, "s", k) for k in ("weight_hh", "bias_hh", "bias_ih")]
        if sync is not None:
            sync.ready([(k, grads[k]) for k in late])
        # input-side weights: dW_ih = d_gi^T X over all frames (layer 0: the packed operand of K1; above: the fp32 outputs of
        # the layer below; zero padded columns)
        for l in range(top, -1, -1):
            for d in ("f", "b", "s"):
                j = (l, d)
                x_in = layers[l]["x"]["f" if d == "f" else "r"]
                rows0, nrows = (t_in(l, d, 0) * B, B) if j == (top, "s") else (0, T * B)
                name = pname(l, d, "weight_ih")
                dw = torch.empty(3 * H, param[name].shape[1], device=dev, dtype=torch.float32)
                _Ops.weight_grad(dgi[j], x_in[rows0:rows0 + nrows], dw, nrows, tensor_core=tc)
                grads[name] = dw
                if sync is not None:
                    sync.ready([(name, dw)])
    return [grads[name] for name, _ in path_parameters(model)]


# ------------------------------------------------------------------------------------------------------------ data parallel
class GradSync:
    """Bucketed all-reduce (sum, then 1 / world_size) of the gradients, issued from inside the backward as soon as a bucket is
    complete: the regressor / heads bucket overlaps the BPTT, the W_hh bucket overlaps the dW_ih GEMMs.  On CUDA tensors the
    collective (NCCL) runs on a side stream; on CPU tensors (gloo, the world-size-2 tests) it runs inline."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.stream = None
        self.bytes = 0
        self.flat = []

    def ready(self, named):
        """named: [(parameter name, gradient tensor)] that are final.  The bucket is flattened and reduced."""
        if self.world == 1 or not named:
            return
        flat = torch.cat([t.reshape(-1) for _, t in named])
        if flat.is_cuda:
            if self.stream is None:
                self.stream = torch.cuda.Stream(device=flat.device)
            ev = torch.cuda.Event()
            ev.record()
            with torch.cuda.stream(self.stream):
                self.stream.wait_event(ev)
                self.dist.all_reduce(flat, group=self.group)
                flat.mul_(1.0 / self.world)
        else:
            self.dist.all_reduce(flat, group=self.group)
            flat.mul_(1.0 / self.world)
        self.bytes += flat.numel() * flat.element_size()
        self.flat.append((flat, [(k, t.numel()) for k, t in named]))

    def finish(self, params: dict):
        """After loss.backward(): waits for the collectives and writes the averaged values into the parameters' .grad."""
        if self.world == 1:
            return
        if self.stream is not None:
            torch.cuda.current_stream().wait_stream(self.stream)
        for flat, pieces in self.flat:
            off = 0
            for name, n in pieces:
                g = params[name].grad
                g.copy_(flat[off:off + n].view_as(g))
                off += n
        self.flat = []


class DataParallel:
    """One replica per GPU (torch.distributed, NCCL); `step(x, masks, loss_fn)` = forward, loss, backward with overlapped gradient
    all-reduce, optimizer step (lib/core/trainer.py:203,235-237 on each rank + the collective the reference does not have)."""

    def __init__(self, model, optimizer, group=None):
        self.model, self.opt = model, optimizer
        self.sync = GradSync(group)

    def step(self, x, loss_fn, dropout_masks=None):
        self.model._grad_sync = self.sync
        self.sync.bytes = 0
        try:
            self.opt.zero_grad(set_to_none=True)
            out = self.model(x, is_train=True, dropout_masks=dropout_masks)
            loss = loss_fn(out[-1])
            loss.backward()
            self.sync.finish(dict(path_parameters(self.model)))
        finally:
            self.model._grad_sync = None
        self.opt.step()
        return loss.detach()
