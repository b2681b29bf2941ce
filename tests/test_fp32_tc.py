"""precision="fp32_tc" checked piece by piece against float64, with bounds the bf16 mode demonstrably fails.

fp32_tc runs the encoder's two big contractions on tensor cores as 3-term bf16 splits: x = hi + lo with hi = RN_bf16(x) and
lo = RN_bf16(x - hi), and x.w ~ hi_x.hi_w + lo_x.hi_w + hi_x.lo_w as ONE bf16 contraction over the K-concatenated operands
[x_hi | x_lo | x_hi] x [W_hi | W_hi | W_lo] (include/tepose_b200.h, TP_PRECISION_BF16X3).  Three pieces of code carry it:

  1. tp_split3_bf16 (csrc/pack.cu) makes the A operand of the input projection: bit-exact against torch's RN_bf16.
  2. tp_gemm_bf16_tc at K = 3 kp over those operands (K1): (a) gemm_check on the exact split operands, (b) against the UNSPLIT
     fp32 product in float64 within the split's representation error + fp32 accumulation; hi-only operands must fail (b).
  3. k_gru_bf16_dual in TP_PRECISION_BF16X3 (K2): (a) a float64 cell whose matmul uses the exact split operands of the fp32
     state, (b) a plain float64 torch.nn.GRU cell at the strict-fp32 tolerance; TP_PRECISION_BF16 must fail (b).

Then: which native path TePose takes in fp32_tc (recorded calls) and where it falls back, and the encoder states and the whole
forward at fp32 grade.  Every bound has a bf16 negative control, so it cannot be loosened into one the bf16 mode passes without a
test failing.  The CPU self-tests show that the float64 references and bounds accept an fp32-accumulated split result and reject
one with lo terms dropped."""
import ctypes
import math

import pytest
import torch

from oracle import synth, torch_ref
from tepose_b200 import _native as nv
from tests.helpers import build_product_model, compare_outputs, gemm_check, oracle_forward

DEV = "cuda:0"
INPUT = synth.INPUT_SIZE                   # 2133
KP = 2176                                  # INPUT rounded up to 64: the packed row width
U_BF16, U_F32 = 2.0 ** -8, 2.0 ** -24
TP_ERR_INVALID, TP_ERR_UNSUPPORTED = -1, -2
GRU_TOL = 2e-5                             # test_gpu_kernels.test_gru_recurrence's strict-fp32 tolerance against float64
GRU_SPLIT_TOL = 4e-6                       # against the float64 cell on the exact split operands: fp32 order + expf / tanhf only
FORWARD_TOL = 5e-6                         # m, vertices and joints of the whole forward against the oracle


# ------------------------------------------------------------------------------------------------------------- splits
def split_hi_lo(x):
    """fp32 x -> (hi, lo) bf16: hi = RN_bf16(x), lo = RN_bf16(x - hi) (x - hi is exact in fp32)."""
    hi = x.to(torch.bfloat16)
    return hi, (x - hi.float()).to(torch.bfloat16)


def split3_rows(x):
    """[x_hi | x_lo | x_hi]: what tp_split3_bf16 writes."""
    hi, lo = split_hi_lo(x)
    return torch.cat([hi, lo, hi], dim=-1)


def split3_weights(w):
    """[W_hi | W_hi | W_lo]: tepose.py's w_ih3 / w_hh3."""
    hi, lo = split_hi_lo(w)
    return torch.cat([hi, hi, lo], dim=-1)


# --------------------------------------------------------------------------------------- K1 against the unsplit product
# Representation error of the three-term split.  With u = 2^-8: x = hi + lo + e, |lo| <= u (1 + u) |x|, |e| <= u^2 |x|, and
# the same for w.  x w - (hi_x hi_w + lo_x hi_w + hi_x lo_w) = hi_x e_w + lo_x lo_w + lo_x e_w + e_x w, so per product
#   |error| <= u^2 (3 + 4 u + 2 u^2) |x| |w|.
SPLIT_REP = U_BF16 ** 2 * (3 + 4 * U_BF16 + 2 * U_BF16 ** 2)
ACC_LAMBDA = 4.0


def split_bound_coeff(k):
    """Coefficient c of the bound |out - x.W^T - b| <= 2^-24 |ref| + c S, S = |x| |W|^T + |b|, for a K1 over k unsplit columns.

    c = SPLIT_REP + ACC_LAMBDA sqrt(3 k) 2^-24: the representation error above (deterministic), plus fp32 accumulation of the 3 k
    exact bf16 products.  The accumulation term is the probabilistic bound of Higham & Mary (SIAM J. Sci. Comput. 41(5), 2019):
    with independent rounding errors the sum of n terms is within lambda sqrt(n) u S except with probability
    <= 2 exp(-lambda^2 / 2) -- 3e-4 per element at lambda = 4, and the real error is far below it, because the partial sums
    are O(sqrt(n)) smaller than S.  The worst-case n u S (gemm_check's term) would be ~17x larger at k = 2176, wide enough to
    admit the hi-only product.  At k = 2176, c = 4.28 2^-16: of order 2^-16 S, as the split promises.  The bf16 mode's error
    is 2^-8 per product, i.e. ~ 2^-8 sqrt(k) |x||w| per element -- several times c S at these operand statistics."""
    return SPLIT_REP + ACC_LAMBDA * math.sqrt(3 * k) * U_F32


def split_gemm_ratio(x, W, bias, out):
    """Worst |out - ref| / bound (NaN -> inf) of out [rows, n] against ref = x.W^T + bias in float64 from the fp32 x [rows, k],
    W [n, k] (unsplit); bound = 2^-24 |ref| + split_bound_coeff(k) S."""
    xd, wd = x.double(), W.double()
    ref = xd @ wd.T
    s = xd.abs() @ wd.abs().T
    if bias is not None:
        ref += bias.double()
        s += bias.double().abs()
    bound = ref.abs() * U_F32 + s * split_bound_coeff(x.shape[1])
    o = out.double()
    err = (o - ref).abs()
    ratio = torch.where(err == 0, torch.zeros_like(err), err / bound)
    return float(ratio.masked_fill(torch.isnan(o) | torch.isnan(ratio), math.inf).max())


def _k1_operands(rows, n, gen, device):
    """Packed-row-like x [rows, KP] ~ N(0, 1) and W [n, KP] ~ U(+-1/sqrt(2048)) (nn.GRU's init at H = 2048), zero past INPUT."""
    x = torch.zeros(rows, KP, device=device)
    x[:, :INPUT] = torch.randn(rows, INPUT, generator=gen, device=device)
    W = torch.zeros(n, KP, device=device)
    k = 2048 ** -0.5
    W[:, :INPUT] = (torch.rand(n, INPUT, generator=gen, device=device) * 2 - 1) * k
    b = (torch.rand(n, generator=gen, device=device) * 2 - 1) * k
    return x, W, b


def test_split_bound_accepts_an_fp32_accumulated_split_product():
    x, W, b = _k1_operands(96, 384, torch.Generator().manual_seed(5), "cpu")
    A3, W3 = split3_rows(x), split3_weights(W)
    out = A3.float() @ W3.float().T + b                  # fp32 accumulation (CPU sgemm) of the exact split products
    r = gemm_check(A3, W3, b, None, False, out)
    assert r.nans == 0 and r.ratio <= 1.0, r
    ratio = split_gemm_ratio(x, W, b, out)
    assert 0.0 < ratio <= 0.5, ratio
    assert split_gemm_ratio(x.double(), W.double(), b, x.double() @ W.double().T + b.double()) == 0.0


@pytest.mark.parametrize("drop", ["all_lo", "x_lo", "w_lo"])
def test_split_bound_rejects_dropped_lo_terms(drop):
    """all_lo: the bf16 mode's product (hi operands only); x_lo / w_lo: one of the three products missing (a lo block of either
    operand written as zeros)."""
    x, W, b = _k1_operands(96, 384, torch.Generator().manual_seed(5), "cpu")
    A3, W3 = split3_rows(x), split3_weights(W)
    if drop in ("all_lo", "x_lo"):
        A3[:, KP:2 * KP] = 0
    if drop in ("all_lo", "w_lo"):
        W3[:, 2 * KP:] = 0
    out = A3.float() @ W3.float().T + b
    assert split_gemm_ratio(x, W, b, out) > 1.5, drop


# --------------------------------------------------------------------------------------------------- K2 references
def gru_ref64(gi, w_hh, b_hh, steps, t_in0=0, t_in_step=1, split=False):
    """States [steps, B, H] (float64, in step order) of the torch.nn.GRU cell from h = 0, driven by gi [T, B, 3H] (the input
    projection incl. b_ih) at t = t_in0 + s t_in_step.  split=False: plain float64.  split=True: the recurrent matmul is the
    float64 value of the BF16X3 contraction the kernel runs -- the fp32 state split as [h_hi | h_lo | h_hi] against
    [W_hi | W_hi | W_lo] -- so what remains between kernel and reference is fp32 accumulation order and expf / tanhf."""
    H = w_hh.shape[1]
    if split:
        wh, wl = (t.double() for t in split_hi_lo(w_hh.float()))
    else:
        wd = w_hh.double()
    b = b_hh.double()
    h = torch.zeros(gi.shape[1], H, dtype=torch.float64, device=gi.device)
    out = []
    for s in range(steps):
        if split:
            hh, hl = (t.double() for t in split_hi_lo(h.float()))
            gh = hh @ wh.T + hl @ wh.T + hh @ wl.T + b
        else:
            gh = h @ wd.T + b
        gx = gi[t_in0 + s * t_in_step].double()
        r = torch.sigmoid(gx[:, :H] + gh[:, :H])
        z = torch.sigmoid(gx[:, H:2 * H] + gh[:, H:2 * H])
        n = torch.tanh(gx[:, 2 * H:] + r * gh[:, 2 * H:])
        h = (1 - z) * n + z * h
        out.append(h)
    return torch.stack(out)


def _gru_fp32_split(gi, w_hh, b_hh, steps, drop_lo=False):
    """The BF16X3 recurrence computed in fp32 on the CPU (exact split products, fp32 sgemm accumulation, fp32 gates)."""
    H = w_hh.shape[1]
    w3 = split3_weights(w_hh).float()
    h = torch.zeros(gi.shape[1], H)
    out = []
    for s in range(steps):
        h3 = split3_rows(h).float()
        if drop_lo:
            h3[:, H:2 * H] = 0
        gh = h3 @ w3.T + b_hh
        gx = gi[s]
        r = torch.sigmoid(gx[:, :H] + gh[:, :H])
        z = torch.sigmoid(gx[:, H:2 * H] + gh[:, H:2 * H])
        n = torch.tanh(gx[:, 2 * H:] + r * gh[:, 2 * H:])
        h = (1 - z) * n + z * h
        out.append(h)
    return torch.stack(out)


def _gru_problem(B, T, H, gen, device):
    k = H ** -0.5
    w = (torch.rand(3 * H, H, generator=gen, device=device) * 2 - 1) * k
    b = (torch.rand(3 * H, generator=gen, device=device) * 2 - 1) * k
    gi = torch.randn(T, B, 3 * H, generator=gen, device=device) * 0.5
    return gi, w, b


def test_gru_ref64_is_torch_nn_gru():
    g = torch.Generator().manual_seed(3)
    B, T, H, F = 3, 5, 64, 24
    gru = torch.nn.GRU(F, H).double()
    x = torch.randn(T, B, F, generator=g, dtype=torch.float64)
    with torch.no_grad():
        y, _ = gru(x)
        gi = x @ gru.weight_ih_l0.T + gru.bias_ih_l0
        got = gru_ref64(gi, gru.weight_hh_l0, gru.bias_hh_l0, T)
        rev = gru_ref64(gi, gru.weight_hh_l0, gru.bias_hh_l0, T, T - 1, -1)
        y_rev, _ = gru(torch.flip(x, [0]))
    assert float((got - y).abs().max()) < 1e-13
    assert float((rev - y_rev).abs().max()) < 1e-13


def test_gru_split_reference_accepts_fp32_split_and_rejects_dropped_lo():
    """The K2 bounds on the CPU: an fp32 evaluation of the split recurrence is within GRU_SPLIT_TOL of reference (a) and GRU_TOL
    of reference (b); with h_lo dropped, or in the bf16 mode's arithmetic (hi operands only), it is outside both."""
    B, T, H = 4, 8, 256
    gi, w, b = _gru_problem(B, T, H, torch.Generator().manual_seed(4), "cpu")
    ref_a = gru_ref64(gi, w, b, T, split=True)
    ref_b = gru_ref64(gi, w, b, T)
    good = _gru_fp32_split(gi, w, b, T)
    ea, eb = float((good - ref_a).abs().max()), float((good - ref_b).abs().max())
    assert ea <= GRU_SPLIT_TOL / 4 and eb <= GRU_TOL / 4, (ea, eb)
    no_lo = _gru_fp32_split(gi, w, b, T, drop_lo=True)
    assert float((no_lo - ref_a).abs().max()) > 4 * GRU_SPLIT_TOL
    assert float((no_lo - ref_b).abs().max()) > 2 * GRU_TOL
    hi_only = gru_ref64(gi, w.to(torch.bfloat16).float(), b, T)          # bf16 weights (the state kept in float64)
    assert float((hi_only - ref_b).abs().max()) > 2 * GRU_TOL


# ======================================================================================================== GPU cases
def _lib():
    return nv.lib()


# --------------------------------------------------------------------------------------------- 1. tp_split3_bf16
def _split3_run(x, rows, k, ld, extra_rows=3):
    """x: CPU fp32 [rows, ld].  Runs tp_split3_bf16 into a NaN-filled [rows + extra_rows, 3k] buffer; returns (rc, buffer bits,
    initial bits)."""
    src = x.to(DEV)
    buf = torch.full(((rows + extra_rows) * 3 * k,), float("nan"), device=DEV, dtype=torch.bfloat16)
    bits0 = buf.view(torch.int16).clone()
    rc = _lib().tp_split3_bf16(nv.vp(src.data_ptr()), ld, rows, k, nv.vp(buf.data_ptr()), nv.stream())
    torch.cuda.synchronize()
    return rc, buf.view(torch.int16).cpu(), bits0.cpu()


def _split3_expect(x, rows, k, ld):
    rc, bits, bits0 = _split3_run(x, rows, k, ld)
    assert rc == 0, _lib().tp_last_error()
    want = split3_rows(x[:, :k]).view(torch.int16).reshape(-1)
    n = rows * 3 * k
    bad = (bits[:n] != want).nonzero()
    assert bad.numel() == 0, f"{bad.numel()} elements differ, first at (row, col) = {divmod(int(bad[0]), 3 * k)}"
    assert torch.equal(bits[n:], bits0[n:]), "rows past `rows` were written"


@pytest.mark.gpu
@pytest.mark.parametrize("rows,k,ld", [(512, KP, KP), (512, KP, KP + 4), (1, 8, 8), (1024, KP, KP), (4096, KP, KP)])
def test_split3_bit_exact(rows, k, ld):
    """[512, 2176]: the packed rows at B = 32, T = 16.  ld = k + 4: a strided source whose 4 pad columns are NaN (read, they
    would show).  [1024 | 4096, 2176]: rows k / 4 > 2048 x 256, the only shapes that reach the grid-stride loop."""
    g = torch.Generator().manual_seed(rows + ld)
    x = torch.full((rows, ld), float("nan"))
    x[:, :k] = torch.randn(rows, k, generator=g) * 3
    _split3_expect(x, rows, k, ld)


@pytest.mark.gpu
def test_split3_special_values():
    """Signed zeros, fp32 subnormals (and lo values that are subnormal), bf16 round-to-even ties, values whose hi rounds up
    (negative lo) and |x| around 1e30.  The library is built without flush-to-zero, so none may be flushed."""
    e = 2.0 ** -8
    vals = [0.0, -0.0, 1e-45, -1e-45, 1e-40, -2.5e-39, 1.1754942e-38, 1.17549435e-38, 1.2e-38, -1.5e-38, 2.0e-38, -3.3e-38,
            1 + e, -(1 + e), 1 + 3 * e, -(1 + 3 * e), 3 * (1 + e), 0.5 * (1 + 5 * e), 1 + 0.75 * 2 * e, 1.9999, -1.9999, 255.9,
            1e30, -1e30, 1.2345678e30, -3.3e30, 7.77e29, 1e-30, math.pi, -math.e]
    x = torch.tensor(vals, dtype=torch.float32)
    g = torch.Generator().manual_seed(9)
    x = torch.cat([x, torch.randn(64 - x.numel(), generator=g)]).repeat(5, 1)
    x[1:] *= torch.tensor([1.0, -1.0, 2.0 ** -100, 2.0 ** 20])[:, None]
    assert bool(torch.isfinite(x).all())
    hi, lo = split_hi_lo(x)
    tiny = 1.17549435e-38
    assert bool(((x.abs() < tiny) & (x != 0)).any()) and bool(((lo.float().abs() < tiny) & (lo != 0)).any())
    assert bool((torch.signbit(x) & (x == 0)).any()) and bool((lo.float() < 0).logical_and(x > 0).any())
    _split3_expect(x, x.shape[0], x.shape[1], x.shape[1])


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["null_src", "null_dst", "k_not_mult_8", "ld_not_mult_4", "src_misaligned", "dst_misaligned",
                                  "no_rows"])
def test_split3_rejects_bad_arguments(case):
    rows, k, ld = 16, 64, 64
    src = torch.randn(rows + 1, ld + 16, device=DEV)
    dst = torch.full((rows * 3 * k + 64,), float("nan"), device=DEV, dtype=torch.bfloat16)
    bits0 = dst.view(torch.int16).clone()
    sp, dp = src.data_ptr(), dst.data_ptr()
    if case == "null_src":
        sp = 0
    elif case == "null_dst":
        dp = 0
    elif case == "k_not_mult_8":
        k = 60
    elif case == "ld_not_mult_4":
        ld = 66
    elif case == "src_misaligned":
        sp += 4
    elif case == "dst_misaligned":
        dp += 8
    elif case == "no_rows":
        rows = 0
    rc = _lib().tp_split3_bf16(nv.vp(sp), ld, rows, k, nv.vp(dp), nv.stream())
    torch.cuda.synchronize()
    assert rc == TP_ERR_INVALID, (case, rc)
    assert b"tp_split3_bf16" in _lib().tp_last_error()
    assert torch.equal(dst.view(torch.int16), bits0)


# ------------------------------------------------------------------------------------------- 2. K1 on the split operands
def _poisoned_out(rows, cols, pad_cols=40, col0=8):
    """NaN [rows + 2, cols + pad_cols] fp32 buffer; the segment writes [:rows, col0:col0 + cols] (a 16-byte aligned window)."""
    buf = torch.full((rows + 2, cols + pad_cols), float("nan"), device=DEV)
    inside = torch.zeros_like(buf, dtype=torch.bool)
    inside[:rows, col0:col0 + cols] = True
    return buf, buf[:rows, col0:col0 + cols], inside


def _k1(A, W, kp, bias, segs):
    """tp_gemm_bf16_tc with `segs` = [(m0, mr, n0, nc)] into poisoned outputs; returns [(out view, buffer, inside mask)]."""
    outs, arr = [], (nv.GemmSeg * len(segs))()
    for i, (m0, mr, n0, nc) in enumerate(segs):
        buf, out, inside = _poisoned_out(mr, nc)
        outs.append((out, buf, inside))
        arr[i] = nv.GemmSeg(m0, mr, n0, nc, nv.vp(out.data_ptr()), buf.shape[1], nv.vp(bias.data_ptr() + 4 * n0), 0, 0, nv.vp(0))
    nv.check(_lib().tp_gemm_bf16_tc(nv.ptr(A), A.shape[0], nv.ptr(W), W.shape[0], kp, arr, len(segs), nv.stream()),
             "tp_gemm_bf16_tc")
    torch.cuda.synchronize()
    return outs


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,H", [(32, 16, 2048), (1, 16, 2048), (17, 5, 256)])
def test_k1_split_operands(B, T, H):
    """The two segments encode_states launches, (0, T B, 0, 6H) and ((T-1) B, B, 6H, 3H), over [x_hi | x_lo | x_hi] (made by
    tp_split3_bf16, as in the forward) and w_ih3 = [W_hi | W_hi | W_lo] [9H, 3 kp]: (a) gemm_check on the exact split operands,
    (b) against the unsplit x.W^T + b in float64.  The same GEMM on hi-only operands (the bf16 mode's K1) must fail (b)."""
    rows = T * B
    x, W, bias = _k1_operands(rows, 9 * H, torch.Generator(DEV).manual_seed(B * 100 + H), DEV)
    x3 = torch.empty(rows, 3 * KP, device=DEV, dtype=torch.bfloat16)
    nv.check(_lib().tp_split3_bf16(nv.ptr(x), KP, rows, KP, nv.ptr(x3), nv.stream()), "tp_split3_bf16")
    W3 = split3_weights(W)
    segs = [(0, rows, 0, 6 * H), ((T - 1) * B, B, 6 * H, 3 * H)]
    report = []
    for (m0, mr, n0, nc), (out, buf, inside) in zip(segs, _k1(x3, W3, 3 * KP, bias, segs)):
        r = gemm_check(x3[m0:m0 + mr], W3[n0:n0 + nc], bias[n0:n0 + nc], None, False, out)
        rb = split_gemm_ratio(x[m0:m0 + mr], W[n0:n0 + nc], bias[n0:n0 + nc], out)
        exact = x[m0:m0 + mr].double() @ W[n0:n0 + nc].double().T + bias[n0:n0 + nc].double()
        split = x3[m0:m0 + mr].double() @ W3[n0:n0 + nc].double().T + bias[n0:n0 + nc].double()
        report.append(f"segment ({m0}, {mr}, {n0}, {nc}): (a) {r.ratio:.3f}  (b) {rb:.3f}   max |gi| {float(exact.abs().max()):.3g}, "
                      f"|out - exact| {float((out.double() - exact).abs().max()):.3g} = split representation "
                      f"{float((split - exact).abs().max()):.3g} + accumulation {float((out.double() - split).abs().max()):.3g}")
        del exact, split
        assert r.nans == 0 and r.ratio <= 1.0, (segs, r)
        assert rb <= 1.0, (segs, rb)
        assert bool(torch.isnan(buf[~inside]).all()), "written outside the segment"
    xh, Wh = x.to(torch.bfloat16), W.to(torch.bfloat16)
    for (m0, mr, n0, nc), (out, buf, inside) in zip(segs, _k1(xh, Wh, KP, bias, segs)):
        r = gemm_check(xh[m0:m0 + mr], Wh[n0:n0 + nc], bias[n0:n0 + nc], None, False, out)
        rb = split_gemm_ratio(x[m0:m0 + mr], W[n0:n0 + nc], bias[n0:n0 + nc], out)
        report.append(f"hi-only ({m0}, {mr}, {n0}, {nc}): (a) {r.ratio:.3f}  (b) {rb:.3f}  <- must exceed 1")
        assert r.nans == 0 and r.ratio <= 1.0, r             # the kernel is right on those operands ...
        assert rb > 1.0, rb                                  # ... and they are not fp32 grade
    print(f"\nK1 fp32_tc B={B} T={T} H={H}: worst |err| / bound\n" + "\n".join(report))


# ---------------------------------------------------------------------------------------------- 3. K2 in BF16X3
def _pack_w3(w):
    """tepose.py's w_hh3: tp_pack_mma_a_bf16 of the [3H, 3H] matrix [W_hi | W_hi | W_lo]."""
    H = w.shape[1]
    w3 = split3_weights(w).float().contiguous()
    out = torch.empty(_lib().tp_pack_mma_a_bytes(3 * H, 3 * H), dtype=torch.uint8, device=DEV)
    nv.check(_lib().tp_pack_mma_a_bf16(nv.ptr(w3), 3 * H, 3 * H, 3 * H, nv.ptr(out), nv.stream()), "tp_pack_mma_a_bf16")
    return out


def _pack_bf16(w):
    out = torch.empty(w.shape, device=DEV, dtype=torch.bfloat16)
    nv.check(_lib().tp_pack_whh_bf16(nv.ptr(w), nv.ptr(out), w.shape[1], nv.stream()), "tp_pack_whh_bf16")
    return out


def _job(gi, col, ldg, w, b, steps, t_in0, t_in_step, y=None, ycol=0, y_lp=None, t_out0=0, t_out_step=1, hf=None, hcol=0,
         h0=None):
    j = nv.GruJob()
    j.gi, j.ldg, j.w_hh, j.b_hh = gi.data_ptr() + 4 * col, ldg, w.data_ptr(), b.data_ptr()
    j.h0 = 0 if h0 is None else h0.data_ptr()
    if y is not None:
        j.y, j.ldy = y.data_ptr() + 4 * ycol, y.shape[-1]
        j.y_lp, j.ldy_lp = y_lp.data_ptr() + 2 * ycol, y_lp.shape[-1]
    if hf is not None:
        j.h_final, j.ld_hf = hf.data_ptr() + 4 * hcol, hf.shape[-1]
    j.steps, j.t_in0, j.t_in_step, j.t_out0, j.t_out_step = steps, t_in0, t_in_step, t_out0, t_out_step
    return j


class _EncoderJobs:
    """The encoder's K2 job set at (B, T0, T1, H): a forward job (T0 steps), a reversed job (T1 steps) -- both reading one
    [Tmax, B, 6H] projection at columns 0 / 3H -- and a single-step job, with NaN-poisoned outputs: y [T, B, H + 24] written at
    column 8, y_lp [T, B, H + 16] bf16 at column 8, and one h_final buffer [B, 3H + 8] written at columns 0 (forward), H (single
    step) and 2H (reversed), as encode_states' h_cat."""
    YC = 8

    def __init__(self, B, T0, T1, H, seed):
        g = torch.Generator(DEV).manual_seed(seed)
        self.B, self.T, self.H = B, (T0, T1), H
        Tm = max(T0, T1)
        gi0, self.w0, self.b0 = _gru_problem(B, Tm, H, g, DEV)
        gi1, self.w1, self.b1 = _gru_problem(B, Tm, H, g, DEV)
        self.gs, self.w2, self.b2 = _gru_problem(B, 1, H, g, DEV)
        self.gi = torch.cat([gi0, gi1], dim=2).contiguous()          # [Tm, B, 6H]
        self.ref = {}
        for split in (True, False):
            self.ref[split] = (gru_ref64(self.gi[..., :3 * H], self.w0, self.b0, T0, split=split),
                               gru_ref64(self.gi[..., 3 * H:], self.w1, self.b1, T1, T1 - 1, -1, split=split),
                               gru_ref64(self.gs, self.w2, self.b2, 1, split=split))

    def run(self, precision, use_slot):
        B, (T0, T1), H, c = self.B, self.T, self.H, self.YC
        pack = _pack_w3 if precision == nv.PRECISION_BF16X3 else _pack_bf16
        w0, w1 = pack(self.w0), pack(self.w1)
        nan = float("nan")
        self.y = [torch.full((t, B, H + 24), nan, device=DEV) for t in (T0, T1)]
        self.ylp = [torch.full((t, B, H + 16), nan, device=DEV, dtype=torch.bfloat16) for t in (T0, T1)]
        self.ylp0 = [t.view(torch.int16).clone() for t in self.ylp]
        self.hf = torch.full((B, 3 * H + 8), nan, device=DEV)
        jobs = [_job(self.gi, 0, 6 * H, w0, self.b0, T0, 0, 1, self.y[0], c, self.ylp[0], hf=self.hf, hcol=0),
                _job(self.gi, 3 * H, 6 * H, w1, self.b1, T1, T1 - 1, -1, self.y[1], c, self.ylp[1], T1 - 1, -1, self.hf, 2 * H),
                _job(self.gs, 0, 3 * H, self.w2, self.b2, 1, 0, 1, hf=self.hf, hcol=H)]
        arr = (nv.GruJob * 3)(*jobs)
        ws = nv.workspace(_lib().tp_gru_workspace_bytes(3, B, H), DEV)
        slot = torch.zeros(256, device=DEV, dtype=torch.int32)
        nv.check(_lib().tp_gru_recurrence_ex(arr, 3, B, H, precision, nv.ptr(ws), ws.numel(),
                                             nv.vp(slot.data_ptr() if use_slot else 0), nv.stream()), "tp_gru_recurrence_ex")
        torch.cuda.synchronize()

    def states(self):
        """(y_fwd [T0,B,H], y_rev [T1,B,H] in output order, h_final [B, 3H]) as float64."""
        H, c = self.H, self.YC
        return self.y[0][..., c:c + H].double(), self.y[1][..., c:c + H].double(), self.hf[:, :3 * H].double()

    def error(self, split):
        """max |kernel - reference| over every state written (y of both directions, the three h_final blocks)."""
        yf, yr, hf = self.states()
        rf, rr, rs = self.ref[split]
        want_hf = torch.cat([rf[-1], rs[-1], rr[-1]], dim=1)
        return max(float((yf - rf).abs().max()), float((yr - torch.flip(rr, [0])).abs().max()), float((hf - want_hf).abs().max()))

    def poison_intact(self):
        H, c = self.H, self.YC
        ok = bool(torch.isnan(self.hf[:, 3 * H:]).all())
        for y in self.y:
            ok &= bool(torch.isnan(y[..., :c]).all()) and bool(torch.isnan(y[..., c + H:]).all())
        for ylp, bits0 in zip(self.ylp, self.ylp0):
            keep = torch.ones(ylp.shape, dtype=torch.bool, device=DEV)
            keep[..., c:c + H] = False
            ok &= torch.equal(ylp.view(torch.int16)[keep], bits0[keep])
        return ok

    def y_lp_is_rounded_y(self):
        H, c = self.H, self.YC
        return all(torch.equal(ylp[..., c:c + H].view(torch.int16), y[..., c:c + H].to(torch.bfloat16).view(torch.int16))
                   for y, ylp in zip(self.y, self.ylp))


K2_CASES = [(32, 16, 16, 2048), (1, 16, 16, 2048), (2, 7, 4, 2048), (3, 5, 7, 128), (8, 4, 6, 1024), (9, 6, 3, 256),
            (17, 5, 8, 256), (31, 4, 2, 1024), (32, 3, 5, 128), (5, 2, 9, 1024)]


@pytest.mark.gpu
@pytest.mark.parametrize("i,B,T0,T1,H", [(i,) + c for i, c in enumerate(K2_CASES)])
def test_k2_bf16x3(i, B, T0, T1, H):
    """k_gru_bf16_dual in TP_PRECISION_BF16X3 (dual<1> at B <= 8, dual<4> at 9..32): (a) against the float64 cell on the exact
    split operands within GRU_SPLIT_TOL, (b) against the plain float64 torch.nn.GRU cell within GRU_TOL.  y_lp is RN_bf16(y) bit
    for bit and nothing outside the outputs' windows is written.  The same jobs in TP_PRECISION_BF16 (same dual kernel,
    bf16 weights and state) must exceed GRU_TOL.  Every other case passes a caller-provided barrier slot."""
    case = _EncoderJobs(B, T0, T1, H, 1000 + i)
    case.run(nv.PRECISION_BF16X3, use_slot=i % 2 == 1)
    ea, eb = case.error(True), case.error(False)
    lp_ok, poison_ok = case.y_lp_is_rounded_y(), case.poison_intact()
    case.run(nv.PRECISION_BF16, use_slot=i % 2 == 1)
    e_bf16 = case.error(False)
    print(f"\nK2 BF16X3 B={B} T=({T0},{T1}) H={H}: (a) {ea:.3g} = {ea / GRU_SPLIT_TOL:.3f} x tol   (b) {eb:.3g} = "
          f"{eb / GRU_TOL:.3f} x tol   bf16 (b) {e_bf16:.3g} = {e_bf16 / GRU_TOL:.1f} x tol")
    assert ea <= GRU_SPLIT_TOL, ea
    assert eb <= GRU_TOL, eb
    assert lp_ok, "y_lp is not RN_bf16(y)"
    assert poison_ok, "written outside the output windows"
    assert case.poison_intact()
    assert e_bf16 > GRU_TOL, e_bf16


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["h0", "one_matmul_job", "three_matmul_jobs", "H96", "B33"])
def test_k2_bf16x3_rejects_unsupported_job_sets(what):
    """BF16X3 is built for exactly two matmul jobs without h0 at B <= 32, H % 128 == 0; anything else is refused, not run."""
    B, H, T = (33 if what == "B33" else 4), (96 if what == "H96" else 128), 3
    g = torch.Generator(DEV).manual_seed(7)
    gi, w, b = _gru_problem(B, T, H, g, DEV)
    w3 = w if H % 128 else _pack_w3(w)
    y = torch.full((T, B, H), float("nan"), device=DEV)
    ylp = torch.full((T, B, H), float("nan"), device=DEV, dtype=torch.bfloat16)
    h0 = torch.zeros(B, H, device=DEV)
    steps = {"one_matmul_job": (T, 1), "three_matmul_jobs": (T, T, T)}.get(what, (T, T, 1))
    jobs = [_job(gi, 0, 3 * H, w3, b, s, 0, 1, y, 0, ylp, h0=h0 if (what == "h0" and i == 0) else None)
            for i, s in enumerate(steps)]
    arr = (nv.GruJob * len(jobs))(*jobs)
    ws = nv.workspace(_lib().tp_gru_workspace_bytes(len(jobs), B, H), DEV)
    rc = _lib().tp_gru_recurrence_ex(arr, len(jobs), B, H, nv.PRECISION_BF16X3, nv.ptr(ws), ws.numel(), nv.vp(0), nv.stream())
    torch.cuda.synchronize()
    assert rc == TP_ERR_UNSUPPORTED, (what, rc)
    assert b"BF16X3" in _lib().tp_last_error()
    assert bool(torch.isnan(y).all()) and bool(torch.isnan(ylp.float()).all())


# ------------------------------------------------------------------------------------------ 4. which path the mode takes
RECORDED = ("tp_split3_bf16", "tp_gemm_bf16_tc", "tp_gemm_f32", "tp_gru_recurrence_ex")


class _RecordingLib:
    """Forwards every call to the real library; the calls named in RECORDED are recorded first (pointers as ints, structure
    arrays as lists of field dicts)."""

    def __init__(self, real, calls):
        self._real, self._calls = real, calls

    def __getattr__(self, name):
        fn = getattr(self._real, name)
        if name not in RECORDED:
            return fn

        def recorded(*args):
            self._calls.append((name, [_decode(a) for a in args]))
            return fn(*args)
        return recorded


def _decode(a):
    if isinstance(a, ctypes.c_void_p):
        return a.value or 0
    if isinstance(a, ctypes.Array):
        return [{f: (getattr(s, f) or 0) for f, _ in type(s)._fields_} for s in a]
    return a


def _recorded(fn, monkeypatch):
    calls = []
    proxy = _RecordingLib(nv.lib(), calls)
    monkeypatch.setattr(nv, "lib", lambda: proxy)
    try:
        with torch.no_grad():
            out = fn()
        torch.cuda.synchronize()
    finally:
        monkeypatch.undo()
    return out, calls


def _by_name(calls, name):
    return [args for n, args in calls if n == name]


def _assert_split_k1(calls, pk, rows_list, B_list, T_list, H):
    """One tp_split3_bf16 per encoder call (on the packed rows, ld = k = kp) feeding one tp_gemm_bf16_tc at K = 3 kp on w_ih3
    with encode_states' two segments; no unsplit fp32 K1 (tp_gemm_f32 at K = kp)."""
    sp, tc = _by_name(calls, "tp_split3_bf16"), _by_name(calls, "tp_gemm_bf16_tc")
    assert len(sp) == len(rows_list) and len(tc) == len(rows_list), (len(sp), len(tc))
    w3 = pk["layers"][0]["w_ih3"]
    for s, t, rows, B, T in zip(sp, tc, rows_list, B_list, T_list):
        assert s[1:4] == [KP, rows, KP], s
        A, a_rows, Wp, w_rows, kp, segs, nseg = t[:7]
        assert (A, a_rows, Wp, w_rows, kp, nseg) == (s[4], rows, w3.data_ptr(), 9 * H, 3 * KP, 2), t[:7]
        got = [(g["m_start"], g["m_rows"], g["n_start"], g["n_cols"]) for g in segs[:nseg]]
        assert got == [(0, T * B, 0, 6 * H), ((T - 1) * B, B, 6 * H, 3 * H)], got
    assert not [a for a in _by_name(calls, "tp_gemm_f32") if a[11] == KP], "an unsplit fp32 K1 ran"


def _recurrence_precisions(calls):
    return [a[4] for a in _by_name(calls, "tp_gru_recurrence_ex")]


@pytest.mark.gpu
def test_fp32_tc_forward_takes_the_split_path(monkeypatch):
    """L = 1, H % 128 == 0, B <= 32, no carried state: tp_split3_bf16 on the packed rows, tp_gemm_bf16_tc at kp = 6528 on w_ih3,
    and tp_gru_recurrence_ex in TP_PRECISION_BF16X3 on the two w_hh3 images."""
    seed, B, T, H = 81, 5, 6, 256
    model, sd = build_product_model(seed, T, 1, H, "fp32_tc", DEV)
    pk = model.encoder.packed()
    x = torch.from_numpy(synth.make_input(seed, B, T)).to(DEV)
    out, calls = _recorded(lambda: model(x)[-1], monkeypatch)
    _assert_split_k1(calls, pk, [T * B], [B], [T], H)
    rec = _by_name(calls, "tp_gru_recurrence_ex")
    assert len(rec) == 1 and rec[0][1:5] == [3, B, H, nv.PRECISION_BF16X3], [r[1:5] for r in rec]
    jobs = rec[0][0]
    assert [jobs[0]["w_hh"], jobs[1]["w_hh"]] == [t.data_ptr() for t in pk["layers"][0]["w_hh3"]]
    assert [j["steps"] for j in jobs] == [T, T, 1]
    ref, _ = oracle_forward(seed, sd, synth.make_input(seed, B, T), 1, H)
    errs = compare_outputs(out, ref, vert_tol=FORWARD_TOL, label="fp32_tc split path")
    print("\nfp32_tc split path", errs)


@pytest.mark.gpu
@pytest.mark.parametrize("L,H,B,T", [(2, 96, 3, 5), (1, 256, 33, 4)])
def test_fp32_tc_forward_fallbacks(L, H, B, T, monkeypatch):
    """L = 2 (or H % 128 != 0): no split operands at all, FP32 recurrences.  B = 33: split K1, FP32 recurrence (fp32_tc batches
    are not grouped into 32-row passes, so K2 sees B = 33).  Each against the oracle at the strict-fp32 tolerances."""
    seed = 82 + L
    model, sd = build_product_model(seed, T, L, H, "fp32_tc", DEV)
    pk = model.encoder.packed()
    x = torch.from_numpy(synth.make_input(seed, B, T)).to(DEV)
    out, calls = _recorded(lambda: model(x)[-1], monkeypatch)
    if L == 2:
        assert not _by_name(calls, "tp_split3_bf16") and not _by_name(calls, "tp_gemm_bf16_tc")
        assert "w_ih3" not in pk["layers"][0] and "w_hh3" not in pk["layers"][0]
        assert _recurrence_precisions(calls) == [nv.PRECISION_FP32] * L
    else:
        _assert_split_k1(calls, pk, [T * B], [B], [T], H)
        assert _recurrence_precisions(calls) == [nv.PRECISION_FP32]
    ref, _ = oracle_forward(seed, sd, synth.make_input(seed, B, T), L, H)
    errs = compare_outputs(out, ref, label=f"fp32_tc fallback L={L} H={H} B={B}")
    print(f"\nfp32_tc fallback L={L} H={H} B={B}", errs)


@pytest.mark.gpu
def test_fp32_tc_live_stream_takes_split_k1_and_fp32_k2(monkeypatch):
    """LiveTePose: the first frame is a one-step window (every K2 job a single step from zero), later frames carry state (h0):
    split K1 and an FP32 recurrence on every frame.  Against the causal oracle at the strict-fp32 tolerances."""
    from tepose_b200.live import LiveTePose
    seed, B, N, H = 83, 1, 4, 256
    model, sd = build_product_model(seed, 16, 1, H, "fp32_tc", DEV)
    pk = model.encoder.packed()
    feats = torch.from_numpy(synth.make_input(seed, B, N))[:, :, :2048]
    live = LiveTePose(model, batch=B, use_graph=False)
    outs, calls = _recorded(lambda: [{k: v.clone().cpu() for k, v in live.step(feats[:, t].to(DEV)).items()} for t in range(N)],
                            monkeypatch)
    Ts = [1] + [2] * (N - 1)
    _assert_split_k1(calls, pk, [T * B for T in Ts], [B] * N, Ts, H)
    assert _recurrence_precisions(calls) == [nv.PRECISION_FP32] * N
    m = torch_ref.SmplModel.synthetic(seed)
    hF = hB = prev = None
    for t in range(N):
        newest = torch.cat([feats[:, t], torch.zeros(B, 85)], dim=1)[:, None]
        if prev is None:
            hFt, hBt, hS = torch_ref.encoder_causal_states(sd, newest, H)
        else:
            hF, hB, _ = torch_ref.encoder_causal_states(sd, prev, H, h0=None if hF is None else (hF, hB))
            hFt, hBt, hS = torch_ref.encoder_causal_states(sd, newest, H, h0=(hF, hB))
        ref = torch_ref.regressor_forward(sd, m, torch_ref.encoder_from_states(sd, hFt, hBt, hS))
        compare_outputs(outs[t], ref, label=f"live fp32_tc frame {t}")
        prev = torch.cat([feats[:, t], ref["theta"]], dim=1)[:, None]


# ------------------------------------------------------------------------------ 5. encoder states and the whole forward
def _encoder_states64(sd, x, H):
    """(h_fwd [B,H], h_rec [B,2H], seq_f [T,B,H], seq_b [T,B,H]) of encode_states from float64 torch.nn.GRU built from the
    state dict: gru_fwd over x, gru_rec's reverse direction over x in original order (x_rec = flip(x)), and gru_rec's forward
    direction one step on the newest frame."""
    xt = x.double().permute(1, 0, 2)

    def gru(prefix, sfx, frames):
        g = torch.nn.GRU(INPUT, H).double().to(x.device)
        g.load_state_dict({f"{n}_l0": torch.as_tensor(sd[f"encoder.{prefix}.{n}_l0{sfx}"]).double()
                           for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")})
        return g(frames)[0]
    with torch.no_grad(), torch.backends.cudnn.flags(enabled=False):
        seq_f = gru("gru_fwd", "", xt)
        seq_b = gru("gru_rec", "_reverse", xt)
        hs = gru("gru_rec", "", xt[-1:])
    return seq_f[-1], torch.cat([hs[0], seq_b[-1]], dim=1), seq_f, seq_b


def test_encoder_states64_matches_the_oracle_encoder():
    """The float64 restatement against oracle/torch_ref's encoder (which is pinned to the reference's goldens), on the CPU."""
    seed, B, T, H = 5, 2, 4, 64
    sd = synth.make_state_dict(seed, 1, H)
    x = torch.from_numpy(synth.make_input(seed, B, T))
    h_fwd, h_rec, seq_f, seq_b = _encoder_states64(sd, x, H)
    gf, gr = torch_ref.build_gru(sd, "gru_fwd", 1, H, False), torch_ref.build_gru(sd, "gru_rec", 1, H, True)
    with torch.no_grad():
        y, _ = gf(x.permute(1, 0, 2))
        y_rec, _ = gr(torch.flip(x.permute(1, 0, 2), [0]))
    assert float((h_fwd - y[-1]).abs().max()) < 1e-5
    assert float((h_rec - y_rec[0]).abs().max()) < 1e-5
    assert float((seq_f - y).abs().max()) < 1e-5
    assert float((seq_b - torch.flip(y_rec[:, :, H:], [0])).abs().max()) < 1e-5


STATE_FACTOR, STATE_FLOOR = 10.0, 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,H", [(32, 16, 2048), (1, 16, 2048), (17, 5, 256), (3, 16, 128)])
def test_encoder_states_at_fp32_grade(B, T, H):
    """encode_states(x, return_states=True) in fp32_tc against float64 torch.nn.GRU: within max(STATE_FACTOR x the strict-fp32
    model's error on the same input, STATE_FLOOR); the bf16 model must exceed that bound.

    Why 10x and not less: fp32_tc's input projection is less exact than the FFMA one, by design rather than by a lost term.  On
    a B200, test_k1_split_operands measures up to ~4e-5 on |gi| <= 3: ~1.3e-5 of split representation error (lo_x lo_w dropped,
    lo rounded: u^2 = 2^-16 per product, SPLIT_REP) and ~3.5e-5 of fp32 accumulation in the tensor core over K = 3 x 2176 (408
    k-steps), against ~1e-6 for the strict-fp32 FFMA K1.  That error carries into every state: the fp32_tc states measure
    6-7.3x the fp32 model's error, while the bf16 model, with no lo terms, measures 550-970x."""
    seed = 90 + H % 1000 + B
    model, sd = build_product_model(seed, T, 1, H, "fp32", DEV)
    x = torch.from_numpy(synth.make_input(seed, B, T)).to(DEV)
    ref = _encoder_states64(sd, x, H)
    errs = {}
    for precision in ("fp32", "fp32_tc", "bf16"):
        model.precision = precision
        with torch.no_grad():
            got = model.encoder.encode_states(x, return_states=True)
        torch.cuda.synchronize()
        errs[precision] = max(float((g.double() - r).abs().max()) for g, r in zip(got, ref))
    bound = max(STATE_FACTOR * errs["fp32"], STATE_FLOOR)
    print(f"\nencoder states B={B} T={T} H={H}: fp32 {errs['fp32']:.3g}  fp32_tc {errs['fp32_tc']:.3g} "
          f"({errs['fp32_tc'] / bound:.3f} x bound {bound:.3g})  bf16 {errs['bf16']:.3g} ({errs['bf16'] / bound:.1f} x bound)")
    assert errs["fp32_tc"] <= bound, errs
    assert errs["bf16"] > bound, errs


@pytest.mark.gpu
@pytest.mark.parametrize("B", [32, 1])
def test_full_forward_at_fp32_grade(B):
    """The full-size forward (L = 1, H = 2048, T = 16) against the oracle with vertices and joints within FORWARD_TOL = 5e-6 m;
    the bf16 model on the same input must exceed it."""
    L, H, T, seed = 1, 2048, 16, 41
    model, sd = build_product_model(seed, T, L, H, "fp32_tc", DEV)
    x = synth.make_input(seed, B, T)
    ref, _ = oracle_forward(seed, sd, x, L, H)
    xd = torch.from_numpy(x).to(DEV)
    with torch.no_grad():
        out = model(xd)[-1]
    errs = compare_outputs(out, ref, vert_tol=FORWARD_TOL, label=f"fp32_tc B={B}")
    model.precision = "bf16"
    with torch.no_grad():
        out_bf16 = model(xd)[-1]
    e_bf16 = max(float((out_bf16[k].cpu() - ref[k]).abs().max()) for k in ("verts", "kp_3d"))
    print(f"\nfull forward B={B}: fp32_tc verts {errs['verts']:.3g} kp_3d {errs['kp_3d']:.3g} (tol {FORWARD_TOL:g})  "
          f"bf16 {e_bf16:.3g} ({e_bf16 / FORWARD_TOL:.1f} x tol)")
    assert e_bf16 > FORWARD_TOL, e_bf16
