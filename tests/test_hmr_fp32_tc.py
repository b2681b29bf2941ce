"""HMR at fp32 grade: precision="fp32_tc" convolutions on split-bf16 tcgen05 GEMMs, from frames to meshes.

An fp32-grade activation of C channels is bf16 [N,H,W,3C], [hi | lo | hi] per pixel (hi = RN_bf16(v), lo = RN_bf16(v - hi));
each folded conv weight is split per tap into [W_hi | W_hi | W_lo], so every convolution is the existing GEMM over the
3C-channel view.  Checked here:
  - CPU: the split pack's column order (that of im2col on the 3C view) and W_hi + W_lo against the float64 folded weight;
  - the new kernels (split crop, NCHW split, split max / average pool) exactly, in NaN-filled buffers larger than their
    output, and their argument checks;
  - the GEMM's TP_GEMM_OUT_SPLIT3 / TP_GEMM_RES_SPLIT3 epilogue on the many-tiles-per-CTA cases of test_hmr_layers.py:
    (hi, lo) = split(v) bit for bit, v the same segment's fp32 output, and v passes gemm_check on the exact split operands;
  - the extractor call by call at 32 and 3 crops, its features against float64 at 1e-4 relative L2 (the bf16 extractor must
    exceed that bound), and the front end (graph, frames, video) bit for bit against the eager paths, and the meshes."""
import collections
import ctypes
import importlib
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import crop_ref, hmr_ref, torch_ref
from tepose_b200 import synthetic as psynth
from tests.helpers import TC_BM, gemm_check
from tests.test_hmr_layers import _check_im2col_call, _avgpool_ratio, _PoisonTorch, _tc_bn, _tiles_per_cta

DEV = "cuda:0"
SEED = 0                                   # bench.py's seed (test_hmr_layers.py's weights and crops)
VIDEO_SEED = 71                            # tests/test_video.py's frames and boxes
GOLD_SEED = 11                             # tests/golden/hmr_N2.npz
FEATURE_TOL = 1e-4                         # relative L2 of the features against float64
TP_ERR_INVALID = -1


# ------------------------------------------------------------------------------------------------------------- splits
def split_hi_lo(x):
    """fp32 x -> (hi, lo) bf16, hi = RN_bf16(x), lo = RN_bf16(x - hi)."""
    hi = x.to(torch.bfloat16)
    return hi, (x - hi.float()).to(torch.bfloat16)


def split3(x):
    """[..., C] fp32 -> [..., 3C] bf16 [hi | lo | hi]."""
    hi, lo = split_hi_lo(x)
    return torch.cat([hi, lo, hi], -1)


def split3_weights(w):
    hi, lo = split_hi_lo(w)
    return torch.cat([hi, hi, lo], -1)


def unsplit(t, C):
    """[..., 3C] split rows -> hi + lo in float64."""
    return t[..., :C].double() + t[..., C:2 * C].double()


def _bits(t):
    return t.contiguous().view(torch.int16)


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm())


# ------------------------------------------------------------------------------------------------------------- CPU
def _conv_bn(cin, cout, k, stride, seed):
    g = torch.Generator().manual_seed(seed)
    conv = torch.nn.Conv2d(cin, cout, k, stride=stride, padding=k // 2, bias=False)
    bn = torch.nn.BatchNorm2d(cout).eval()
    with torch.no_grad():
        conv.weight.copy_(torch.randn(cout, cin, k, k, generator=g) * (2.0 / (k * k * cout)) ** 0.5)
        bn.weight.uniform_(0.5, 1.5, generator=g); bn.bias.normal_(generator=g)
        bn.running_mean.normal_(generator=g); bn.running_var.uniform_(0.5, 2.0, generator=g)
    return conv, bn


@pytest.mark.parametrize("cin,cout,k,stride,cin_pad", [(3, 64, 7, 2, 4), (8, 16, 3, 2, None), (64, 256, 1, 1, None)])
def test_split_pack_column_order_and_precision(cin, cout, k, stride, cin_pad):
    """The split pack holds [W_hi | W_hi | W_lo] per tap in the column order of im2col over the 3C-channel view, W_hi + W_lo
    reproduces the float64 folded weight within 2^-16 relative, and the padded columns are zero.  Then the convolution as
    im2col rows of [x_hi | x_lo | x_hi] times the pack (float64 products) matches the float64 conv + BatchNorm at fp32 grade,
    where the bf16 pack does not."""
    from tepose_b200.hmr import _fold, _fold_split3
    conv, bn = _conv_bn(cin, cout, k, stride, cin * k)
    w3, b = _fold_split3(conv, bn, cin_pad=cin_pad)
    C = cin_pad or cin
    K = k * k * 3 * C
    assert w3.dtype == torch.bfloat16 and w3.shape == (cout, (K + 63) // 64 * 64) and w3.shape[1] % 64 == 0
    assert bool((w3[:, K:] == 0).all())
    scale = bn.weight.detach().double() / torch.sqrt(bn.running_var.double() + bn.eps)
    w64 = torch.zeros(cout, C, k, k, dtype=torch.float64)
    w64[:, :cin] = conv.weight.detach().double() * scale[:, None, None, None]
    w64 = w64.permute(0, 2, 3, 1)                                                # (ky, kx, c)
    taps = w3[:, :K].view(cout, k, k, 3, C)
    hi, lo = taps[..., 0, :], taps[..., 2, :]
    assert torch.equal(_bits(taps[..., 1, :]), _bits(hi))                          # W_hi twice
    assert torch.equal(_bits(hi), _bits(w64.to(torch.bfloat16)))
    assert float(((hi.double() + lo.double()) - w64).abs().max()) <= 2.0 ** -16 * float(w64.abs().max())
    assert bool(((hi.double() + lo.double() - w64).abs() <= 2.0 ** -16 * w64.abs()).all())
    # the convolution through im2col on the 3C view
    x = torch.randn(2, cin, 11, 9, generator=torch.Generator().manual_seed(5))
    xp = torch.zeros(2, C, 11, 9)
    xp[:, :cin] = x
    x3 = split3(xp.permute(0, 2, 3, 1)).double().permute(0, 3, 1, 2)              # [N, 3C, H, W]
    cols = F.unfold(x3, k, padding=k // 2, stride=stride)                          # (c, ky, kx)
    L = cols.shape[-1]
    cols = cols.view(2, 3 * C, k * k, L).permute(0, 3, 2, 1).reshape(2, L, K)      # -> (ky, kx, c)
    got = cols @ w3[:, :K].double().T + b.double()
    with torch.no_grad():
        want = bn.double()(conv.double()(x.double())).permute(0, 2, 3, 1).reshape(2, L, cout)
    rel = _rel(got, want)
    w1, b1 = _fold(conv.float(), bn.float(), cin_pad=cin_pad)
    cols1 = F.unfold(xp.permute(0, 2, 3, 1).to(torch.bfloat16).double().permute(0, 3, 1, 2), k, padding=k // 2, stride=stride)
    cols1 = cols1.view(2, C, k * k, L).permute(0, 3, 2, 1).reshape(2, L, k * k * C)
    rel_bf16 = _rel(cols1 @ w1[:, :k * k * C].double().T + b1.double(), want)
    print(f"conv through the split pack: {rel:.3g}, through the bf16 pack: {rel_bf16:.3g} relative L2")
    assert rel < 2e-5 and rel_bf16 > 30 * rel, (rel, rel_bf16)


def test_hmr_precision_modes():
    with pytest.raises(ValueError):
        psynth.build_synthetic_hmr(3, "cpu", precision="fp32")
    m = psynth.build_synthetic_hmr(3, "cpu", precision="fp32_tc")
    assert m.precision == "fp32_tc" and m.stem_channels == 12
    assert psynth.build_synthetic_hmr(3, "cpu").stem_channels == 4


# ------------------------------------------------------------------------------------------------------------- kernels
def _guarded(n, dtype):
    """A NaN buffer of n elements plus a 64-element tail that must stay NaN."""
    buf = torch.full((n + 64,), float("nan"), device=DEV, dtype=dtype)
    return buf, buf[:n]


def _table(rows):
    from tepose_b200.hmr import make_crop_table
    return make_crop_table(np.array(rows, np.float64), DEV)


def _crop_split(frames, table, N, out):
    from tepose_b200 import _native as nv
    F_, H, W, _ = frames.shape
    return nv.lib().tp_crop_normalize_split3(nv.ptr(frames), F_, H, W, nv.ptr(table), N, nv.ptr(out), nv.stream())


def _crops_split_ref(frames, rows):
    """split(normalize(crop(...))) with channel 3 zero: [N, 224, 224, 12] bf16."""
    out = torch.zeros(len(rows), 224, 224, 4)
    for i, (f, *r) in enumerate(rows):
        out[i, ..., :3] = torch.from_numpy(crop_ref.normalize(crop_ref.crop(frames[int(f)], *r)))
    return split3(out)


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(97, 131), (1080, 1920)])
@pytest.mark.parametrize("N", [1, 3, 32])
def test_split_crop_is_bit_exact(H, W, N):
    frames = crop_ref.sample_frames(VIDEO_SEED + H, 2, H, W)
    rows = crop_ref.sample_boxes(VIDEO_SEED, 2, H, W)
    rows = rows[:N] if N != 1 else [rows[1]]
    out = torch.full((N + 2, 224, 224, 12), float("nan"), dtype=torch.bfloat16, device=DEV)
    from tepose_b200 import _native as nv
    nv.check(_crop_split(torch.from_numpy(frames).to(DEV), _table(rows), N, out), "tp_crop_normalize_split3")
    torch.cuda.synchronize()
    want = _crops_split_ref(frames, rows)
    got = out[:N].cpu()
    for i in range(N):
        diff = int((_bits(got[i]) != _bits(want[i])).sum())
        assert diff == 0, (i, rows[i], diff)
    assert bool(torch.isnan(out[N:].float()).all())


@pytest.mark.gpu
def test_split_crop_rejects_invalid_arguments_and_zeroes_bad_frames_under_capture():
    from tepose_b200 import _native as nv
    L = nv.lib()
    frames = torch.zeros(2, 20, 30, 3, dtype=torch.uint8, device=DEV)
    table = _table([(1, 10.0, 10.0, 8.0, 8.0, 1.2), (0, 5.0, 5.0, 8.0, 8.0, 1.0)])
    bad_frame = _table([(0, 10.0, 10.0, 8.0, 8.0, 1.2), (2, 5.0, 5.0, 8.0, 8.0, 1.0)])
    out = torch.full((3, 224, 224, 12), float("nan"), dtype=torch.bfloat16, device=DEV)
    f, t, o, st = nv.ptr(frames), nv.ptr(table), nv.ptr(out), nv.stream()
    raw = ctypes.c_void_p
    cases = {
        "null frames": (None, 2, 20, 30, t, 2, o), "null crops": (f, 2, 20, 30, None, 2, o), "null out": (f, 2, 20, 30, t, 2, None),
        "N = 0": (f, 2, 20, 30, t, 0, o), "N > 65535": (f, 2, 20, 30, t, 65536, o), "F = 0": (f, 0, 20, 30, t, 2, o),
        "H = 0": (f, 2, 0, 30, t, 2, o), "W < 0": (f, 2, 20, -30, t, 2, o),
        "out 8 bytes off alignment": (f, 2, 20, 30, t, 2, raw(out.data_ptr() + 8)),
        "crops 2 bytes off alignment": (f, 2, 20, 30, raw(table.data_ptr() + 2), 2, o),
        "frame index == F": (f, 2, 20, 30, nv.ptr(bad_frame), 2, o), "frame index >= F (F = 1)": (f, 1, 20, 30, t, 2, o),
    }
    for name, (fp, F_, H, W, tp, N, op) in cases.items():
        assert L.tp_crop_normalize_split3(fp, F_, H, W, tp, N, op, st) == TP_ERR_INVALID, name
        assert b"tp_crop_normalize_split3" in L.tp_last_error(), name
    torch.cuda.synchronize()
    assert bool(torch.isnan(out.float()).all())
    # under capture: boxes rewritten between replays are followed; a frame index gone bad gives zeros for that crop
    H, W = 97, 131
    fr_np = crop_ref.sample_frames(VIDEO_SEED, 2, H, W)
    rows = crop_ref.sample_boxes(VIDEO_SEED + 1, 2, H, W)
    a = rows[1:3]
    fr = torch.from_numpy(fr_np).to(DEV)
    table = _table(a)
    out = torch.zeros(2, 224, 224, 12, dtype=torch.bfloat16, device=DEV)
    nv.check(_crop_split(fr, table, 2, out))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        nv.check(_crop_split(fr, table, 2, out))
    table.copy_(_table([(2,) + tuple(a[0][1:]), rows[5]]))
    g.replay()
    torch.cuda.synchronize()
    assert bool((_bits(out[0]) == 0).all())
    assert torch.equal(_bits(out[1].cpu()), _bits(_crops_split_ref(fr_np, [rows[5]])[0]))


@pytest.mark.gpu
def test_nchw_to_nhwc_split3_is_bit_exact():
    from tepose_b200 import _native as nv
    L = nv.lib()
    g = torch.Generator(DEV).manual_seed(3)
    x = torch.randn(32, 3, 224, 224, generator=g, device=DEV) * 3
    x[0, 0, 0, :4] = torch.tensor([0.0, -0.0, 1e-30, -3.0e38])                    # zero signs, a subnormal-range lo, a large value
    buf, out = _guarded(32 * 224 * 224 * 12, torch.bfloat16)
    nv.check(L.tp_nchw_to_nhwc_split3(nv.ptr(x), nv.ptr(out), 32, 3, 224, 224, 4, nv.stream()))
    xp = torch.zeros(32, 224, 224, 4, device=DEV)
    xp[..., :3] = x.permute(0, 2, 3, 1)
    assert torch.equal(_bits(out), _bits(split3(xp).view(-1)))
    assert bool(torch.isnan(buf[out.numel():]).all())
    o = nv.ptr(out)
    for args in [(None, o, 1, 3, 8, 8, 4), (nv.ptr(x), None, 1, 3, 8, 8, 4), (nv.ptr(x), o, 0, 3, 8, 8, 4),
                 (nv.ptr(x), o, 1, 3, 8, 8, 2), (nv.ptr(x), o, 1, 3, 0, 8, 4)]:
        assert L.tp_nchw_to_nhwc_split3(*args, nv.stream()) == TP_ERR_INVALID, args


def _split_rows(shape, gen, negative=False):
    """A canonical split tensor [..., 3C] of fp32 values (as the GEMM epilogue writes them), and those values."""
    v = torch.randn(*shape, generator=gen, device=DEV) * 2
    if negative:
        v = -(v.abs() + 0.01)
    return split3(v), v


def _maxpool_split_ref(x3, C):
    """float64 restatement: per window the first (ky, kx) position whose hi + lo is the largest; its (hi, lo) pair."""
    N, H, W, _ = x3.shape
    val = unsplit(x3, C).permute(0, 3, 1, 2)                                         # [N, C, H, W] float64
    pad = F.pad(val, (1, 1, 1, 1), value=-math.inf)
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    win = pad.unfold(2, 3, 2).unfold(3, 3, 2)[:, :, :Ho, :Wo].reshape(N, C, Ho, Wo, 9)
    arg = win.argmax(-1)                                                             # first maximal index
    ky, kx = arg // 3, arg % 3
    hh = torch.arange(Ho, device=DEV)[None, None, :, None] * 2 - 1 + ky
    ww = torch.arange(Wo, device=DEV)[None, None, None, :] * 2 - 1 + kx
    n = torch.arange(N, device=DEV)[:, None, None, None]
    c = torch.arange(C, device=DEV)[None, :, None, None]
    hi, lo = x3[n, hh, ww, c], x3[n, hh, ww, C + c]
    return torch.cat([hi, lo, hi], 1).permute(0, 2, 3, 1).contiguous()             # [N, Ho, Wo, 3C]


@pytest.mark.gpu
@pytest.mark.parametrize("size,negative", [(112, False), (112, True), (113, True), (14, False)])
def test_maxpool_split3_is_bit_exact(size, negative):
    """[32,112,112,64] is the stem's max pool at 32 crops; 113: a last window over the bottom/right edge; all-negative input
    shows a border window that took the padding as 0.  Ties: the 14 x 14 case repeats values across pixels."""
    from tepose_b200 import _native as nv
    g = torch.Generator(DEV).manual_seed(size + negative)
    N = 32 if size > 100 else 2
    x3, _ = _split_rows((N, size, size, 64), g, negative)
    if size == 14:
        x3 = x3[:, ::2].repeat_interleave(2, 1).contiguous()                        # equal values in adjacent rows
    Ho = (size - 1) // 2 + 1
    buf, out = _guarded(N * Ho * Ho * 192, torch.bfloat16)
    nv.check(nv.lib().tp_maxpool3x3s2_nhwc_split3(nv.ptr(x3), nv.ptr(out), N, size, size, 64, nv.stream()))
    want = _maxpool_split_ref(x3, 64)
    assert torch.equal(_bits(out), _bits(want.view(-1)))
    assert bool(torch.isnan(buf[out.numel():]).all())
    # the represented value is the max of the represented values of the window
    assert torch.equal(unsplit(out.view(N, Ho, Ho, 192), 64),
                       F.max_pool2d(unsplit(x3, 64).permute(0, 3, 1, 2), 3, 2, 1).permute(0, 2, 3, 1))


@pytest.mark.gpu
def test_avgpool_split3_within_its_fp32_bound():
    from tepose_b200 import _native as nv
    g = torch.Generator(DEV).manual_seed(49)
    x3, _ = _split_rows((32, 49, 2048), g)
    x3 = split3((unsplit(x3, 2048).float() + 0.5))
    buf, out = _guarded(32 * 2048, torch.float32)
    nv.check(nv.lib().tp_avgpool_nhwc_split3(nv.ptr(x3), nv.ptr(out), 32, 49, 2048, nv.stream()))
    torch.cuda.synchronize()
    # the bound of test_hmr_layers._avgpool_ratio on the represented values hi + lo (exact in fp32)
    assert _avgpool_ratio(unsplit(x3, 2048).float(), out.view(32, 2048)) <= 1.0
    assert bool(torch.isnan(buf[out.numel():]).all())


@pytest.mark.gpu
def test_split_pools_reject_invalid_arguments():
    from tepose_b200 import _native as nv
    L = nv.lib()
    a = torch.zeros(2 * 14 * 14 * 48 + 8, dtype=torch.bfloat16, device=DEV)
    o = torch.full((2 * 7 * 7 * 48 + 8,), float("nan"), dtype=torch.bfloat16, device=DEV)
    f = torch.full((2 * 16,), float("nan"), device=DEV)
    pa, po, st = nv.ptr(a), nv.ptr(o), nv.stream()
    off = ctypes.c_void_p(a.data_ptr() + 2)
    for args in [(None, po, 2, 14, 14, 16), (pa, None, 2, 14, 14, 16), (pa, po, 2, 14, 14, 12), (pa, po, 0, 14, 14, 16),
                 (off, po, 2, 14, 14, 16), (pa, ctypes.c_void_p(o.data_ptr() + 8), 2, 14, 14, 16)]:
        assert L.tp_maxpool3x3s2_nhwc_split3(*args, st) == TP_ERR_INVALID, args
    for args in [(None, nv.ptr(f), 2, 49, 16), (pa, None, 2, 49, 16), (pa, nv.ptr(f), 2, 0, 16), (pa, nv.ptr(f), 2, 49, 0)]:
        assert L.tp_avgpool_nhwc_split3(*args, st) == TP_ERR_INVALID, args
    torch.cuda.synchronize()
    assert bool(torch.isnan(o).all()) and bool(torch.isnan(f).all())


# ------------------------------------------------------------------------------------------------------------- GEMM
INT_VIEW = {torch.bfloat16: torch.int16, torch.float32: torch.int32}


def _split_operands(rows, w_rows, k, seed):
    """A = [x_hi | x_lo | x_hi] [rows, 3k] and W = [W_hi | W_hi | W_lo] [w_rows, 3k] of fp32 x ~ N(0,1), w ~ N(0, 1/k)."""
    g = torch.Generator(DEV).manual_seed(seed)
    x = torch.randn(rows, k, generator=g, device=DEV)
    w = torch.randn(w_rows, k, generator=g, device=DEV) / k ** 0.5
    return split3(x).contiguous(), split3_weights(w).contiguous(), g


class _Seg:
    """One segment and its NaN-filled output buffer, larger than the segment (`extra` rows, ldc past the 3 n_cols of a split
    output).  split: output in split layout; its fp32 twin (split=False) writes v.  res: None, "bf16" or "split"."""

    def __init__(self, g, m_start, m_rows, n_start, n_cols, *, relu=False, split=True, bf16=False, bias=True, res=None,
                 ldc=None, extra=3, res_data=None, bias_data=None):
        from tepose_b200 import _native as nv
        self.m_start, self.m_rows, self.n_start, self.n_cols, self.relu, self.split = m_start, m_rows, n_start, n_cols, relu, split
        self.dtype = torch.bfloat16 if (split or bf16) else torch.float32
        width = 3 * n_cols if split else n_cols
        ldc = ldc or width + 24
        self.ldc = ldc
        self.buf = torch.full(((m_rows + extra) * ldc,), float("nan"), device=DEV, dtype=self.dtype)
        self.bits0 = self.buf.view(INT_VIEW[self.dtype]).clone()
        self.inside = torch.zeros(self.buf.shape, device=DEV, dtype=torch.bool)
        self.inside[:m_rows * ldc].view(m_rows, ldc)[:, :width] = True
        self.out = self.buf[:m_rows * ldc].view(m_rows, ldc)[:, :width]
        self.bias = bias_data if bias_data is not None else (torch.randn(n_cols, generator=g, device=DEV) if bias else None)
        flags = (nv.GEMM_RELU if relu else 0) | (nv.GEMM_OUT_SPLIT3 if split else (nv.GEMM_OUT_BF16 if bf16 else 0))
        self.res_buf, self.residual, ldr = None, None, 0
        if res is not None:
            if res_data is None:
                v = torch.randn(m_rows, n_cols, generator=g, device=DEV)
                ldr = 3 * n_cols + 8 if res == "split" else n_cols + 8
                res_data = torch.zeros(m_rows, ldr, device=DEV, dtype=torch.bfloat16)
                res_data[:, :3 * n_cols if res == "split" else n_cols] = split3(v) if res == "split" else v.to(torch.bfloat16)
            self.res_buf, ldr = res_data, res_data.shape[1]
            self.residual = unsplit(res_data, n_cols).float() if res == "split" else res_data[:, :n_cols]
            if res == "split":
                flags |= nv.GEMM_RES_SPLIT3
        self.res_kind = res
        self.seg = nv.GemmSeg(m_start, m_rows, n_start, n_cols, nv.vp(self.buf.data_ptr()), ldc, nv.ptr(self.bias), flags, ldr,
                              nv.ptr(self.res_buf))

    def twin(self):
        """The same segment with fp32 output (same bias, same residual rows)."""
        return _Seg(None, self.m_start, self.m_rows, self.n_start, self.n_cols, relu=self.relu, split=False, res=self.res_kind,
                    res_data=self.res_buf, bias_data=self.bias, bias=self.bias is not None)


def _launch(A, W, segs):
    from tepose_b200 import _native as nv
    arr = (nv.GemmSeg * len(segs))(*[s.seg for s in segs])
    rc = nv.lib().tp_gemm_bf16_tc(nv.ptr(A), A.shape[0], nv.ptr(W), W.shape[0], A.shape[1], arr, len(segs), nv.stream())
    torch.cuda.synchronize()
    return rc


def _run_split_and_check(A, W, segs):
    """Runs the segments, then their fp32 twins in a launch of the same shape (same tile width and tile order), and checks
    every split segment: (hi, lo, hi) = split(v) bit for bit, v within gemm_check on the exact operands, nothing written
    outside any segment."""
    from tepose_b200 import _native as nv
    nv.check(_launch(A, W, segs), "tp_gemm_bf16_tc")
    twins = [s.twin() for s in segs]
    nv.check(_launch(A, W, twins), "tp_gemm_bf16_tc (fp32 twins)")
    bn = _tc_bn([(s.m_rows, s.n_cols) for s in segs])
    for i, (s, t) in enumerate(zip(segs, twins)):
        v = t.out
        r = gemm_check(A[s.m_start:s.m_start + s.m_rows], W[s.n_start:s.n_start + s.n_cols], s.bias, s.residual, s.relu, v)
        tile = (r.row // TC_BM * TC_BM, r.col // bn * bn)
        assert r.nans == 0 and r.ratio <= 1.0, f"segment {i}: worst ratio {r.ratio:.3g} ({r.nans} NaN), tile {tile}, BN {bn}"
        if s.split:
            assert torch.equal(_bits(s.out), _bits(split3(v))), f"segment {i}: split output differs from split(v)"
        else:
            assert torch.equal(s.out.float(), v.to(s.dtype).float()), f"segment {i}"
        for x in (s, t):
            changed = (x.buf.view(INT_VIEW[x.dtype]) != x.bits0) & ~x.inside
            assert not bool(changed.any()), f"segment {i}: {int(changed.sum())} elements written outside the segment"
    return bn


MANY_ROWS, MANY_COLS = 1000, 25008     # 8 m-tiles (last one 104 rows) x 131 n-tiles of 192 (last one 48 columns) = 1048 tiles


@pytest.mark.gpu
@pytest.mark.parametrize("k3", [192, 4032])
@pytest.mark.parametrize("relu,res", [(False, None), (True, None), (False, "split"), (True, "split"), (True, "bf16")])
def test_split_gemm_many_tiles_per_cta(k3, relu, res):
    """1048 tiles on the persistent CTAs (>= 8 per CTA) with TP_GEMM_OUT_SPLIT3, alone and with ReLU and a bf16 or split
    residual.  k3 = 3 x 64: one 192-wide contraction; 3 x 1344: the smem ring wraps many times per tile."""
    A, W, g = _split_operands(MANY_ROWS, MANY_COLS + 48, k3 // 3, k3 + 8 * relu + len(res or ""))
    s = _Seg(g, 0, MANY_ROWS, 16, MANY_COLS, relu=relu, res=res)
    bn = _run_split_and_check(A, W, [s])
    assert bn == 192 and _tiles_per_cta([(MANY_ROWS, MANY_COLS)], bn)[1] >= 8


@pytest.mark.gpu
@pytest.mark.parametrize("past_one_wave", [0, 1])
def test_split_gemm_tile_width_switch(past_one_wave):
    sm = torch.cuda.get_device_properties(DEV).multi_processor_count
    rows = (sm + past_one_wave) * TC_BM - 40
    A, W, g = _split_operands(rows, 320, 256, 21 + past_one_wave)
    for relu, res in ((False, None), (True, "split")):
        s = _Seg(g, 0, rows, 64, 128, relu=relu, res=res)
        assert _run_split_and_check(A, W, [s]) == (192 if past_one_wave else 128)


@pytest.mark.gpu
def test_split_gemm_eight_segments():
    """Eight segments mixing split and plain outputs, split and bf16 residuals, a single-row segment and an odd n_start."""
    A, W, g = _split_operands(1500, 1200, 64, 31)
    spec = [(0, 300, 0, 160, dict(relu=True, res="split")),
            (37, 129, 160, 64, dict(split=False, bf16=True)),
            (200, 1, 304, 16, dict(relu=True)),
            (511, 400, 96, 336, dict(res="split")),
            (1000, 500, 640, 560, dict(relu=True, split=False, res="split")),
            (5, 128, 1184, 16, dict(bias=False, res="bf16")),
            (777, 255, 17, 48, dict(relu=True, res="split")),
            (1400, 100, 400, 48, dict(split=False, bf16=True, res="split"))]
    segs = [_Seg(g, m0, mr, n0, nc, **kw) for m0, mr, n0, nc, kw in spec]
    _run_split_and_check(A, W, segs)


@pytest.mark.gpu
def test_split_gemm_rejects_bad_layouts():
    from tepose_b200 import _native as nv
    A, W, g = _split_operands(128, 64, 64, 41)
    cases = {}
    s = _Seg(g, 0, 128, 0, 64, ldc=3 * 64 - 8)                       # ldc < 3 n_cols
    cases["ldc < 3 n_cols"] = s
    s = _Seg(g, 0, 128, 0, 64, ldc=3 * 64 + 4)                       # ldc % 8 != 0
    cases["ldc % 8"] = s
    s = _Seg(g, 0, 128, 0, 64)
    s.seg.out = s.buf.data_ptr() + 8                                 # out 8 bytes off 16-byte alignment
    cases["unaligned out"] = s
    s = _Seg(g, 0, 128, 0, 64, res="split")
    s.seg.ldr = 3 * 64 - 8                                           # ldr < 3 n_cols
    cases["ldr < 3 n_cols"] = s
    s = _Seg(g, 0, 128, 0, 64)
    s.seg.flags |= nv.GEMM_RES_SPLIT3                                # split residual flag without a residual
    cases["no residual"] = s
    for name, s in cases.items():
        assert _launch(A, W, [s]) == TP_ERR_INVALID, name
        assert b"split" in nv.lib().tp_last_error(), name
        assert bool(torch.isnan(s.buf.float()).all()), name


# ------------------------------------------------------------------------------------------------------------- extractor
RECORDED = ("tp_nchw_to_nhwc_split3", "tp_im2col_nhwc_bf16", "tp_gemm_bf16_tc", "tp_maxpool3x3s2_nhwc_split3",
            "tp_avgpool_nhwc_split3")


class _RecordingLib:
    def __init__(self, real, calls):
        self._real, self._calls = real, calls

    def __getattr__(self, name):
        fn = getattr(self._real, name)
        if name not in RECORDED:
            return fn

        def recorded(*args):
            from tepose_b200 import _native as nv
            dec = []
            for a in args:
                if isinstance(a, ctypes.c_void_p):
                    a = a.value or 0
                elif isinstance(a, ctypes.Array):
                    a = [{f: (getattr(s, f) or 0) for f, _ in nv.GemmSeg._fields_} for s in a]
                dec.append(a)
            self._calls.append((name, dec))
            return fn(*args)
        return recorded


def _record_extractor(model, x, monkeypatch):
    from tepose_b200 import _native as nv
    hmr_mod = importlib.import_module("tepose_b200.hmr")
    registry = {x.data_ptr(): x}
    pk = model.conv_packed_split3()
    for wb in [pk["stem"]] + [e[k] for e in pk["blocks"] for k in ("c1", "c2", "c3", "down") if e[k] is not None]:
        for t in wb:
            registry[t.data_ptr()] = t
    calls = []
    proxy = _RecordingLib(nv.lib(), calls)
    monkeypatch.setattr(nv, "lib", lambda: proxy)
    monkeypatch.setattr(hmr_mod, "torch", _PoisonTorch(registry))
    with torch.no_grad():
        xf = model.feature_extractor(x)
    torch.cuda.synchronize()
    monkeypatch.undo()
    return xf, calls, registry, pk


def _tensor(registry, p, shape, dtype):
    assert p in registry, f"pointer {p:#x} is not a tensor the extractor allocated or a packed weight"
    t = registry[p]
    assert t.dtype == dtype and t.numel() == math.prod(shape), (t.dtype, dtype, tuple(t.shape), shape)
    return t.view(shape)


def _wire(calls, pk, x, N, size=224):
    """HMR's bottleneck structure in split layout, followed through the recorded calls by pointer identity."""
    from tepose_b200 import _native as nv
    names, it = [], iter(enumerate(calls))

    def take(name, label):
        i, (got, args) = next(it)
        assert got == name, (i, label, got, name)
        names.append(label)
        return args

    def gemm(label, a, rows, wb, relu, residual=0):
        A, a_rows, Wp, w_rows, kp, segs, nseg = take("tp_gemm_bf16_tc", label)[:7]
        w, b = wb
        cout = w.shape[0]
        assert (A, a_rows, Wp, w_rows, kp, nseg) == (a, rows, w.data_ptr(), cout, w.shape[1], 1), label
        s = segs[0]
        assert (s["m_start"], s["m_rows"], s["n_start"], s["n_cols"], s["ldc"]) == (0, rows, 0, cout, 3 * cout), (label, s)
        flags = (nv.GEMM_RELU if relu else 0) | nv.GEMM_OUT_SPLIT3 | (nv.GEMM_RES_SPLIT3 if residual else 0)
        assert s["bias"] == b.data_ptr() and s["flags"] == flags, (label, s)
        assert s["residual"] == residual and s["ldr"] == (3 * cout if residual else 0), (label, s)
        return s["out"]

    H = W = size
    a = take("tp_nchw_to_nhwc_split3", "stem.nchw_to_nhwc")
    assert a[0] == x.data_ptr() and a[2:7] == [N, 3, H, W, 4], a
    kp = pk["stem"][0].shape[1]
    assert kp == 640
    a2 = take("tp_im2col_nhwc_bf16", "stem.im2col")
    assert a2[0] == a[1] and a2[2:11] == [N, H, W, 12, 7, 7, 2, 3, kp], a2
    H, W = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    y = gemm("stem.conv1", a2[1], N * H * W, pk["stem"], True)
    a = take("tp_maxpool3x3s2_nhwc_split3", "stem.maxpool")
    assert a[0] == y and a[2:6] == [N, H, W, 64], a
    cur, Cin = a[1], 64
    H, W = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    blocks = [f"layer{li + 1}.{bi}" for li, n in enumerate((3, 4, 6, 3)) for bi in range(n)]
    for name, e in zip(blocks, pk["blocks"]):
        planes, s = e["planes"], e["stride"]
        t1 = gemm(f"{name}.conv1", cur, N * H * W, e["c1"], True)
        Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
        a = take("tp_im2col_nhwc_bf16", f"{name}.im2col")
        assert a[0] == t1 and a[2:11] == [N, H, W, 3 * planes, 3, 3, s, 1, 27 * planes], (name, a)
        t2 = gemm(f"{name}.conv2", a[1], N * Ho * Wo, e["c2"], True)
        if e["down"] is not None:
            src = cur
            if s != 1:
                a = take("tp_im2col_nhwc_bf16", f"{name}.downsample.im2col")
                assert a[0] == cur and a[2:11] == [N, H, W, 3 * Cin, 1, 1, s, 0, 3 * Cin], (name, a)
                src = a[1]
            res = gemm(f"{name}.downsample", src, N * Ho * Wo, e["down"], False)
        else:
            res = cur
        cur = gemm(f"{name}.conv3", t2, N * Ho * Wo, e["c3"], True, residual=res)
        H, W, Cin = Ho, Wo, planes * 4
    a = take("tp_avgpool_nhwc_split3", "avgpool")
    assert a[0] == cur and a[2:5] == [N, H * W, Cin], a
    assert next(it, None) is None
    return names


def _check_split_gemm_call(registry, args):
    """gemm_check on the exact split operands, with the represented output hi + lo in fp32 (exact there).  The bound stays
    valid: the lo rounding adds at most 2^-18 |v|, and gemm_check's accumulation term KP 2^-23 S leaves (KP - 2) 2^-24 S
    >= 2^-18 S above the worst-case fp32 accumulation for every KP >= 66 (here KP >= 192); S >= |v|."""
    A, a_rows, Wp, w_rows, kp, segs, nseg = args[:7]
    A = _tensor(registry, A, (a_rows, kp), torch.bfloat16)
    W = _tensor(registry, Wp, (w_rows, kp), torch.bfloat16)
    s = segs[0]
    mr, nc = s["m_rows"], s["n_cols"]
    o = _tensor(registry, s["out"], (mr, s["ldc"]), torch.bfloat16)
    # a split the epilogue wrote: the third block repeats hi, and hi is a nearest bf16 to v = hi + lo (|lo| <= |v - RN(v)|;
    # RN(hi + lo) itself may be hi's neighbour when lo rounded to exactly half an ulp and the tie goes to even)
    v = unsplit(o, nc)
    canonical = torch.equal(_bits(o[:, :nc]), _bits(o[:, 2 * nc:3 * nc])) and \
        bool((o[:, nc:2 * nc].double().abs() <= (v - v.float().to(torch.bfloat16).double()).abs()).all())
    b = _tensor(registry, s["bias"], (nc,), torch.float32)
    r = unsplit(_tensor(registry, s["residual"], (mr, s["ldr"]), torch.bfloat16), nc).float() if s["residual"] else None
    return gemm_check(A, W, b, r, bool(s["flags"] & 1), unsplit(o, nc).float()), canonical, (mr, nc), kp


@pytest.fixture(scope="module")
def hmr_pair():
    """The same synthetic weights as precision "fp32_tc" and "bf16"."""
    return (psynth.build_synthetic_hmr(SEED, DEV, precision="fp32_tc"), psynth.build_synthetic_hmr(SEED, DEV))


def _float64_features(model, x):
    sd = {k: v.double() for k, v in model.state_dict().items() if v.is_floating_point() and not k.startswith("smpl.")}
    with torch.no_grad():
        return hmr_ref.feature_extractor(sd, x.double())


@pytest.mark.gpu
@pytest.mark.parametrize("crops", [32, 3])
def test_every_native_call_of_the_split_extractor(hmr_pair, crops, monkeypatch):
    model, model_bf16 = hmr_pair
    x = torch.from_numpy(psynth.make_image_batch(SEED, crops)).to(DEV)
    xf, calls, registry, pk = _record_extractor(model, x, monkeypatch)
    counts = collections.Counter(name for name, _ in calls)
    assert counts == {"tp_nchw_to_nhwc_split3": 1, "tp_im2col_nhwc_bf16": 20, "tp_gemm_bf16_tc": 53,
                      "tp_maxpool3x3s2_nhwc_split3": 1, "tp_avgpool_nhwc_split3": 1}, counts
    names = _wire(calls, pk, x, crops)

    bad, report, worst = [], [], collections.defaultdict(float)
    for label, (name, args) in zip(names, calls):
        if name == "tp_nchw_to_nhwc_split3":
            xp, yp, N, C, H, W, CP = args[:7]
            y = _tensor(registry, yp, (N, H, W, 3 * CP), torch.bfloat16)
            want = torch.zeros(N, H, W, CP, device=DEV)
            want[..., :C] = x.permute(0, 2, 3, 1)
            if not torch.equal(_bits(y), _bits(split3(want))):
                bad.append(f"{label}: not bit-exact")
        elif name == "tp_im2col_nhwc_bf16":
            if not _check_im2col_call(registry, args):
                bad.append(f"{label}: not bit-exact against F.unfold")
        elif name == "tp_maxpool3x3s2_nhwc_split3":
            inp, outp, N, H, W, C = args[:6]
            x3 = _tensor(registry, inp, (N, H, W, 3 * C), torch.bfloat16)
            out = _tensor(registry, outp, (N, (H - 1) // 2 + 1, (W - 1) // 2 + 1, 3 * C), torch.bfloat16)
            if not torch.equal(_bits(out), _bits(_maxpool_split_ref(x3, C))):
                bad.append(f"{label}: not bit-exact against the float64 restatement")
        elif name == "tp_avgpool_nhwc_split3":
            inp, outp, N, HW, C = args[:5]
            out = _tensor(registry, outp, (N, C), torch.float32)
            assert out.data_ptr() == xf.data_ptr()
            ratio = _avgpool_ratio(unsplit(_tensor(registry, inp, (N, HW, 3 * C), torch.bfloat16), C).float(), out)
            report.append(f"{label:24s} ratio {ratio:.3f}")
            if not ratio <= 1.0:
                bad.append(f"{label}: avg-pool error ratio {ratio:.3g}")
        else:
            r, canonical, (rows, cout), kp = _check_split_gemm_call(registry, args)
            bn = _tc_bn([(rows, cout)])
            tiles, per_cta = _tiles_per_cta([(rows, cout)], bn)
            layer = label.split(".")[0]
            worst[layer] = max(worst[layer], r.ratio)
            report.append(f"{label:24s} rows {rows:6d} cout {cout:4d} kp {kp:5d}  BN {bn}  tiles {tiles:4d} "
                          f"(<= {per_cta:2d} per CTA)  worst ratio {r.ratio:.3f}")
            if r.nans or not r.ratio <= 1.0 or not canonical:
                bad.append(f"{label}: worst ratio {r.ratio:.3g} ({r.nans} NaN) at row {r.row} col {r.col}, canonical split {canonical}")
    print(f"\nHMR fp32_tc feature_extractor, {crops} crops: every native call against float64 (ratio = |err| / bound)")
    print("\n".join(report))
    print("worst GEMM ratio per layer: " + ", ".join(f"{k} {v:.3f}" for k, v in worst.items()))
    assert not bad, "\n".join(bad)

    # the features against the float64 restatement on the same fp32 input; the bf16 extractor must exceed the bound
    want = _float64_features(model, x)
    rel = _rel(xf, want)
    with torch.no_grad():
        rel_bf16 = _rel(model_bf16.feature_extractor(x), want)
    print(f"features against float64, {crops} crops: fp32_tc {rel:.3g}, bf16 {rel_bf16:.3g} relative L2")
    assert rel <= FEATURE_TOL < rel_bf16, (rel, rel_bf16)


@pytest.mark.gpu
def test_split_extractor_against_the_reference_golden():
    """tests/golden/hmr_N2.npz: features of the unmodified reference HMR (fp32); the bf16 extractor is 3.1e-3 away from it."""
    import os
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "hmr_N2.npz"))
    model = psynth.build_synthetic_hmr(GOLD_SEED, DEV, precision="fp32_tc")
    x = torch.from_numpy(psynth.make_image_batch(GOLD_SEED, 2)).to(DEV)
    with torch.no_grad():
        xf = model.feature_extractor(x)
        xf2, out = model(x, return_features=True)
    assert torch.equal(xf, xf2)
    rel = _rel(xf, torch.from_numpy(z["xf"]))
    print(f"\nfp32_tc features against the reference golden: {rel:.3g} relative L2")
    assert rel <= FEATURE_TOL, rel
    assert set(out[0]) == {"theta", "verts", "kp_2d", "kp_3d"}
    for k in ("verts", "kp_3d"):
        err = float((out[0][k].cpu() - torch.from_numpy(z[k])).abs().max())
        assert err < 1e-4, (k, err)


# ------------------------------------------------------------------------------------------------------------- front end
@pytest.mark.gpu
def test_graphed_split_extractor_is_bit_identical_to_eager(hmr_pair):
    from tepose_b200.graph import GraphedHMRFeatures
    model = hmr_pair[0]
    x = torch.from_numpy(psynth.make_image_batch(SEED, 32)).to(DEV)
    with torch.no_grad():
        eager = model.feature_extractor(x).clone()
    g = GraphedHMRFeatures(model, 32)
    got = g(x)
    torch.cuda.synchronize()
    assert g.launches_per_replay == 76
    assert torch.equal(got, eager)


@pytest.fixture(scope="module")
def video_models():
    """HMR fp32_tc and bf16 with test_video.py's weights; TePose T4 L1 H64 fp32_tc, VIBE L2 H32."""
    from tepose_b200.synthetic import build_synthetic_model, build_synthetic_vibe
    model, sd = build_synthetic_model(VIDEO_SEED, 4, 1, 64, "fp32_tc", DEV)
    vibe, sd_v = build_synthetic_vibe(VIDEO_SEED, 4, 2, 32, True, False, True, "fp32", DEV)
    return (psynth.build_synthetic_hmr(VIDEO_SEED, DEV, precision="fp32_tc"), psynth.build_synthetic_hmr(VIDEO_SEED, DEV),
            model, vibe, sd, sd_v, torch_ref.SmplModel.synthetic(VIDEO_SEED))


@pytest.mark.gpu
def test_split_features_from_frames_equal_feature_extractor_on_the_reference_crops(video_models):
    hmr = video_models[0]
    H, W = 1080, 1920
    frames = crop_ref.sample_frames(VIDEO_SEED + 5, 2, H, W)
    rows = crop_ref.sample_boxes(VIDEO_SEED + 5, 2, H, W)[:5]
    with torch.no_grad():
        got = hmr.features_from_frames(torch.from_numpy(frames).to(DEV), rows)
        nchw = np.stack([crop_ref.normalize(crop_ref.crop(frames[f], *r)) for f, *r in rows]).transpose(0, 3, 1, 2)
        want = hmr.feature_extractor(torch.from_numpy(np.ascontiguousarray(nchw)).to(DEV))
    assert got.shape == (5, 2048)
    assert torch.equal(got, want)


def _clip(B, N, H=180, W=320):
    frames = crop_ref.sample_frames(VIDEO_SEED + 9, N, H, W)
    crops = np.zeros((B, N, 6))
    for b in range(B):
        for t in range(N):
            crops[b, t] = (0, W * (0.3 + 0.4 * b) + 3.7 * t, H * 0.5 - 1.3 * t, 60 + 2 * t, 120 - t, 1.2)
    return frames, crops


@pytest.mark.gpu
def test_video_with_split_hmr_equals_windowed_run_and_meshes_reach_fp32_grade(video_models):
    """VideoTePose (fp32_tc HMR and TePose) equals WindowedTePose.run on the features the split HMR extracts, bit for bit; its
    vertices against the oracle chain on float64 features (hmr_ref in float64 on the restated crops -> the oracle's windowed
    TePose with VIBE bootstrap) are within 1e-4 m and at most 1/30 of the bf16 HMR chain's error."""
    from tepose_b200 import VideoTePose
    from tepose_b200.stream import WindowedTePose
    hmr, hmr_bf16, model, vibe, sd, sd_v, m = video_models
    J = m.J_regressor_h36m
    B, T = 2, 4
    N = T + 3
    frames, crops = _clip(B, N)
    fr = torch.from_numpy(frames).to(DEV)
    with torch.no_grad():
        feats = torch.stack([hmr.features_from_frames(fr[t:t + 1], crops[:, t]) for t in range(N)], 1)
    want = WindowedTePose(model, vibe, J_regressor=J, batch=B).run(feats)
    got = VideoTePose(hmr, model, vibe, J_regressor=J, batch=B).run(fr, torch.from_numpy(crops).to(DEV))
    for k in ("theta", "verts", "kp_2d", "kp_3d", "rotmat"):
        assert torch.equal(got[k], want[k]), (k, float((got[k] - want[k]).abs().max()))
    got_bf16 = VideoTePose(hmr_bf16, model, vibe, J_regressor=J, batch=B).run(fr, crops)

    nchw = np.stack([np.stack([crop_ref.normalize(crop_ref.crop(frames[t], *crops[b, t, 1:])) for t in range(N)])
                     for b in range(B)]).transpose(0, 1, 4, 2, 3)                      # [B, N, 3, 224, 224]
    f64 = _float64_features(hmr, torch.from_numpy(np.ascontiguousarray(nchw)).reshape(B * N, 3, 224, 224).to(DEV))
    ref = torch_ref.windowed_stream(sd_v, dict(n_layers=2, hidden=32, add_linear=True, bidirectional=False, use_residual=True),
                                    sd, m, f64.float().cpu().reshape(B, N, 2048), T, 1, 64, J_regressor=J)
    err = float((got["verts"].cpu() - ref["verts"]).abs().max())
    err_bf16 = float((got_bf16["verts"].cpu() - ref["verts"]).abs().max())
    print(f"\nmax vertex error against the float64-feature chain: fp32_tc {err:.3g} m, bf16 HMR {err_bf16:.3g} m")
    assert err <= 1e-4 and err <= err_bf16 / 30, (err, err_bf16)
