"""Shared test helpers: synthetic base_data directory, model construction, golden files, comparisons."""
import ast
import collections
import contextlib
import math
import os
import tempfile

import numpy as np
import torch

from oracle import synth, torch_ref

FORWARD_OUTPUTS = ("theta", "verts", "kp_2d", "kp_3d", "rotmat")
TC_BM = 128                                # k_gemm_bf16_tc tile rows
U_OUT = {torch.bfloat16: 2.0 ** -8, torch.float32: 2.0 ** -24}


@contextlib.contextmanager
def base_data_cwd(seed=0):
    """cwd with data/base_data/* (the reference's asset paths are cwd-relative:
    lib/core/config.py:31)."""
    old = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        synth.write_base_data(os.path.join(tmp, "data", "base_data"), seed)
        os.chdir(tmp)
        try:
            yield tmp
        finally:
            os.chdir(old)


def build_product_model(seed, seqlen, n_layers, hidden, precision="fp32", device="cpu"):
    from tepose_b200.synthetic import build_synthetic_model
    return build_synthetic_model(seed, seqlen, n_layers, hidden, precision, device)


def oracle_forward(seed, sd, x, n_layers, hidden, is_train=False, use_h36m=False):
    m = torch_ref.SmplModel.synthetic(seed)
    return torch_ref.tepose_forward(sd, m, torch.as_tensor(x), n_layers, hidden, is_train=is_train,
                                    J_regressor=m.J_regressor_h36m if use_h36m else None), m


def load_forward_golden(path):
    """(cfg, outputs, cut) of a forward golden file (oracle/make_golden.py:save_forward).  Files of large batches keep a seeded
    sample of each mesh (verts_idx[r]: the vertex indices kept for output row r); cut(out) reduces a forward's outputs, torch
    tensors on any device, to what the file holds."""
    z = np.load(path)
    cfg = ast.literal_eval(str(z["cfg"]))
    gold = {k: z[k] for k in FORWARD_OUTPUTS}
    idx = torch.from_numpy(z["verts_idx"].astype(np.int64)) if "verts_idx" in z.files else None

    def cut(out):
        if idx is None:
            return out
        v = out["verts"]
        return dict(out, verts=torch.gather(v, 1, idx.to(v.device)[..., None].expand(-1, -1, v.shape[-1])))
    return cfg, gold, cut


def aa_to_R(aa):
    return torch_ref.batch_rodrigues_smplx(torch.as_tensor(aa, dtype=torch.float32).reshape(-1, 3))


def compare_outputs(got, ref, vert_tol=1e-4, rot_tol=1e-5, kp2d_tol=1e-3, label=""):
    """Tolerances of SURVEY.md 8(c): verts / joints max-abs <= 1e-4 m (fp32), rotmat <= 1e-5,
    theta compared after mapping the axis-angle part through aa -> R, kp_2d <= 1e-3."""
    g = {k: (v.detach().cpu() if torch.is_tensor(v) else torch.as_tensor(v)) for k, v in got.items()}
    r = {k: (v.detach().cpu() if torch.is_tensor(v) else torch.as_tensor(v)) for k, v in ref.items()}
    errs = {}
    for k in ("verts", "kp_3d", "rotmat", "kp_2d"):
        assert g[k].shape == r[k].shape, (label, k, g[k].shape, r[k].shape)
        errs[k] = float((g[k] - r[k]).abs().max())
    tg, tr = g["theta"].reshape(-1, 85), r["theta"].reshape(-1, 85)
    errs["theta_cam_shape"] = float(torch.cat([tg[:, :3] - tr[:, :3], tg[:, 75:] - tr[:, 75:]], 1).abs().max())
    errs["theta_pose_as_R"] = float((aa_to_R(tg[:, 3:75]) - aa_to_R(tr[:, 3:75])).abs().max())
    assert errs["verts"] <= vert_tol, (label, errs)
    assert errs["kp_3d"] <= vert_tol, (label, errs)
    assert errs["rotmat"] <= rot_tol, (label, errs)
    assert errs["kp_2d"] <= kp2d_tol, (label, errs)
    assert errs["theta_cam_shape"] <= rot_tol * 10, (label, errs)
    assert errs["theta_pose_as_R"] <= rot_tol * 10, (label, errs)
    return errs


GemmCheck = collections.namedtuple("GemmCheck", "ratio row col nans")


def gemm_check(A, W, bias, residual, relu, out, max_bytes=2 << 30):
    """out [rows, Cout] (bf16 or fp32, may be a strided window) against ref = act(A . W^T + bias + residual) in float64 from the
    exact bf16 operands A [rows, KP], W [Cout, KP] (bias fp32 [Cout] or None, residual bf16 [rows, Cout] or None).

    Bound per element: |out - ref| <= u |ref| + KP 2^-23 S,  S = |A| |W|^T + |bias| + |residual|.  u is one rounding of the
    output (2^-8 bf16, 2^-24 fp32); the second term covers fp32 accumulation of the KP exact products and the two epilogue adds.
    ReLU is 1-Lipschitz, so the bound holds after it.  Runs on the inputs' device, chunked over rows so that the float64
    temporaries stay around `max_bytes`.  Returns the worst |out - ref| / bound, where it is, and the NaN count of `out`."""
    rows, kp = A.shape
    cout = W.shape[0]
    assert W.shape[1] == kp and tuple(out.shape) == (rows, cout), (A.shape, W.shape, out.shape)
    u, acc = U_OUT[out.dtype], kp * 2.0 ** -23
    w = W.double()
    wa = w.abs()
    b = bias.double() if bias is not None else None
    per_row = 8 * (2 * kp + 8 * cout)
    chunk = max(TC_BM, (max_bytes - 16 * cout * kp) // per_row)
    worst, where, nans = 0.0, (0, 0), 0
    for r0 in range(0, rows, chunk):
        a = A[r0:r0 + chunk].double()
        ref, s = a @ w.T, a.abs() @ wa.T
        del a
        if b is not None:
            ref += b
            s += b.abs()
        if residual is not None:
            r = residual[r0:r0 + chunk].double()
            ref += r
            s += r.abs()
            del r
        if relu:
            ref.clamp_(min=0.0)
        bound = ref.abs().mul_(u).add_(s, alpha=acc)
        del s
        o = out[r0:r0 + chunk].double()
        nan = torch.isnan(o)
        nans += int(nan.sum())
        err = (o - ref).abs_()
        del o, ref
        ratio = torch.where(err == 0, torch.zeros_like(err), err / bound)        # 0 / 0 -> 0, x / 0 -> inf
        ratio.masked_fill_(nan | torch.isnan(ratio), math.inf)
        i = int(ratio.argmax())
        if float(ratio.view(-1)[i]) > worst or r0 == 0:
            worst, where = float(ratio.view(-1)[i]), (r0 + i // cout, i % cout)
    return GemmCheck(worst, where[0], where[1], nans)
