"""HMR ResNet-50 feature extractor checked call by call at the benchmark's batch (32 crops), and the tcgen05 GEMM at its edges.

Every native call HMR.feature_extractor makes is recorded (a proxy around tepose_b200._native.lib()) and checked against a float64
reference computed from that call's own inputs, with every buffer the extractor allocates NaN-poisoned first.  An error in one
tile of one layer therefore cannot hide behind the bf16 drift accumulated over 53 convolutions (tests/test_hmr.py compares the
final features only, at 2 and 5 crops, where one persistent CTA runs at most 4 GEMM tiles; at 32 crops it runs up to 22).

The GEMM comparator (gemm_check) bounds every element by one rounding of the output plus fp32 accumulation over the inner
dimension; test_gemm_check_* shows on CPU that it accepts an fp32-accumulated result and rejects small, plausible kernel bugs,
so the bound cannot be loosened into something vacuous without a test failing."""
import collections
import ctypes
import importlib
import itertools
import math

import pytest
import torch
import torch.nn.functional as F

from tepose_b200 import synthetic as psynth
from tests.helpers import TC_BM, gemm_check

DEV = "cuda:0"
SEED = 0                                   # bench.py's seed: the same weights and crops the benchmark times
INT_VIEW = {torch.bfloat16: torch.int16, torch.float32: torch.int32}


# ---------------------------------------------------------------------------------------------------------------- comparator
def _selftest_operands(relu):
    g = torch.Generator().manual_seed(7)
    rows, cout, kp = 1000, 256, 576                  # a layer1 3x3 conv: 8 m-tiles with a ragged last one (104 rows)
    A = torch.randn(rows, kp, generator=g).to(torch.bfloat16)
    W = (torch.randn(cout, kp, generator=g) / kp ** 0.5).to(torch.bfloat16)
    bias = torch.randn(cout, generator=g)
    R = torch.randn(rows, cout, generator=g).to(torch.bfloat16)

    def result(k=kp, b=bias, r=R):                   # fp32 accumulation (CPU sgemm), fp32 epilogue, as the kernel computes it
        y = A[:, :k].float() @ W[:, :k].float().T + b + r.float()
        return y.clamp_min(0.0) if relu else y
    return A, W, bias, R, result


@pytest.mark.parametrize("relu", [False, True])
def test_gemm_check_accepts_an_fp32_accumulated_result(relu):
    A, W, bias, R, result = _selftest_operands(relu)
    y = result()
    for out in (y.to(torch.bfloat16), y):
        r = gemm_check(A, W, bias, R, relu, out)
        assert r.nans == 0 and 0.0 < r.ratio <= 1.0, (out.dtype, r)
    r = gemm_check(A, W, None, None, relu, (A.float() @ W.float().T).clamp_min(0.0 if relu else -math.inf).to(torch.bfloat16))
    assert r.ratio <= 1.0, r


@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("mutation", ["zero_tile", "swap_rows", "bias_shift", "residual_missing", "last_kblock", "nan"])
def test_gemm_check_rejects_a_wrong_tile(mutation, relu):
    """Each mutation is a kernel bug that would still leave the final HMR features within a loose norm bound."""
    A, W, bias, R, result = _selftest_operands(relu)
    y = result()
    if mutation == "zero_tile":                      # one 128 x 64 tile never written (or written with zeros)
        y[256:384, 64:128] = 0.0
    elif mutation == "swap_rows":                    # two adjacent rows of one tile exchanged (a TMEM lane / row mapping slip)
        y[[300, 301]] = y[[301, 300]]
    elif mutation == "bias_shift":                   # bias applied one column off
        y = result(b=torch.roll(bias, -1))
    elif mutation == "residual_missing":             # shortcut not added in one tile
        y[384:512, 128:192] = result(r=torch.zeros_like(R))[384:512, 128:192]
    elif mutation == "last_kblock":                  # the last 64-wide k-block never accumulated
        y = result(k=A.shape[1] - 64)
    elif mutation == "nan":
        y[999, 255] = float("nan")
    r = gemm_check(A, W, bias, R, relu, y.to(torch.bfloat16))
    assert r.ratio > 1.0, (mutation, r)
    if mutation == "nan":
        assert r.nans == 1 and (r.row, r.col) == (999, 255) and r.ratio == math.inf


# ------------------------------------------------------------------------------------------------ recording the extractor
def _tc_bn(shapes):
    """The tile width tp_gemm_bf16_tc's dispatch picks for segments of (m_rows, n_cols): 192 past one wave of 128 x 128 tiles."""
    tiles128 = sum(math.ceil(m / TC_BM) * math.ceil(n / 128) for m, n in shapes)
    return 192 if tiles128 > torch.cuda.get_device_properties(DEV).multi_processor_count else 128


def _tiles_per_cta(shapes, bn):
    tiles = sum(math.ceil(m / TC_BM) * math.ceil(n / bn) for m, n in shapes)
    return tiles, math.ceil(tiles / min(tiles, torch.cuda.get_device_properties(DEV).multi_processor_count))


class _PoisonTorch:
    """The `torch` tepose_b200/hmr.py sees: `empty` returns NaN-filled tensors and registers them by data pointer, so a tile
    a kernel never writes reads back as NaN rather than as stale, correct data left by the caching allocator."""

    def __init__(self, registry):
        self._registry = registry

    def __getattr__(self, name):
        return getattr(torch, name)

    def empty(self, *size, **kw):
        t = torch.empty(*size, **kw).fill_(float("nan"))
        self._registry[t.data_ptr()] = t
        return t


RECORDED = ("tp_nchw_to_nhwc_bf16", "tp_im2col_nhwc_bf16", "tp_gemm_bf16_tc", "tp_maxpool3x3s2_nhwc_bf16", "tp_avgpool_nhwc_bf16")


class _RecordingLib:
    """Forwards every call to the real library; the HMR kernels' arguments are recorded first (pointers as ints, GemmSeg
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
    from tepose_b200 import _native as nv
    if isinstance(a, ctypes.c_void_p):
        return a.value or 0
    if isinstance(a, ctypes.Array):
        return [{f: (getattr(s, f) or 0) for f, _ in nv.GemmSeg._fields_} for s in a]
    return a


def _record_extractor(model, x, monkeypatch):
    from tepose_b200 import _native as nv
    hmr_mod = importlib.import_module("tepose_b200.hmr")     # (the package exports the function `hmr` under that name)
    registry = {x.data_ptr(): x}
    pk = model.conv_packed()
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
    """The registered tensor at device pointer p, viewed as `shape` (it must be exactly that large)."""
    assert p in registry, f"pointer {p:#x} is not a tensor the extractor allocated or a packed weight"
    t = registry[p]
    assert t.dtype == dtype and t.numel() == math.prod(shape), (t.dtype, dtype, tuple(t.shape), shape)
    return t.view(shape)


def _wire(calls, pk, x, N, size=224):
    """Follows HMR.feature_extractor's bottleneck structure through the recorded calls by pointer identity; returns the name
    of every call."""
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
        assert (s["m_start"], s["m_rows"], s["n_start"], s["n_cols"], s["ldc"]) == (0, rows, 0, cout, cout), (label, s)
        assert s["bias"] == b.data_ptr() and s["flags"] == (nv.GEMM_RELU if relu else 0) | nv.GEMM_OUT_BF16, (label, s)
        assert s["residual"] == residual and s["ldr"] == (cout if residual else 0), (label, s)
        return s["out"]

    H = W = size
    a = take("tp_nchw_to_nhwc_bf16", "stem.nchw_to_nhwc")
    assert a[0] == x.data_ptr() and a[2:7] == [N, 3, H, W, 4], a
    kp = pk["stem"][0].shape[1]
    a2 = take("tp_im2col_nhwc_bf16", "stem.im2col")
    assert a2[0] == a[1] and a2[2:11] == [N, H, W, 4, 7, 7, 2, 3, kp], a2
    H, W = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    y = gemm("stem.conv1", a2[1], N * H * W, pk["stem"], True)
    a = take("tp_maxpool3x3s2_nhwc_bf16", "stem.maxpool")
    assert a[0] == y and a[2:6] == [N, H, W, 64], a
    cur, Cin = a[1], 64
    H, W = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    blocks = [f"layer{li + 1}.{bi}" for li, n in enumerate((3, 4, 6, 3)) for bi in range(n)]
    assert len(blocks) == len(pk["blocks"])
    for name, e in zip(blocks, pk["blocks"]):
        planes, s = e["planes"], e["stride"]
        t1 = gemm(f"{name}.conv1", cur, N * H * W, e["c1"], True)
        Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
        a = take("tp_im2col_nhwc_bf16", f"{name}.im2col")
        assert a[0] == t1 and a[2:11] == [N, H, W, planes, 3, 3, s, 1, 9 * planes], (name, a)
        t2 = gemm(f"{name}.conv2", a[1], N * Ho * Wo, e["c2"], True)
        if e["down"] is not None:
            src = cur
            if s != 1:
                a = take("tp_im2col_nhwc_bf16", f"{name}.downsample.im2col")
                assert a[0] == cur and a[2:11] == [N, H, W, Cin, 1, 1, s, 0, Cin], (name, a)
                src = a[1]
            res = gemm(f"{name}.downsample", src, N * Ho * Wo, e["down"], False)
        else:
            res = cur
        cur = gemm(f"{name}.conv3", t2, N * Ho * Wo, e["c3"], True, residual=res)
        H, W, Cin = Ho, Wo, planes * 4
    a = take("tp_avgpool_nhwc_bf16", "avgpool")
    assert a[0] == cur and a[2:5] == [N, H * W, Cin], a
    assert next(it, None) is None
    return names


def _check_gemm_call(registry, args):
    A, a_rows, Wp, w_rows, kp, segs, nseg = args[:7]
    A = _tensor(registry, A, (a_rows, kp), torch.bfloat16)
    W = _tensor(registry, Wp, (w_rows, kp), torch.bfloat16)
    out = []
    for s in segs[:nseg]:
        m0, mr, n0, nc = s["m_start"], s["m_rows"], s["n_start"], s["n_cols"]
        dt = torch.bfloat16 if s["flags"] & 2 else torch.float32
        o = _tensor(registry, s["out"], (mr, s["ldc"]), dt)[:, :nc]
        b = _tensor(registry, s["bias"], (nc,), torch.float32) if s["bias"] else None
        r = _tensor(registry, s["residual"], (mr, s["ldr"]), torch.bfloat16)[:, :nc] if s["residual"] else None
        out.append((gemm_check(A[m0:m0 + mr], W[n0:n0 + nc], b, r, bool(s["flags"] & 1), o), (mr, nc), kp))
    return out


def _check_im2col_call(registry, args):
    inp, outp, N, H, W, C, kh, kw, s, pad, KP = args[:11]
    x = _tensor(registry, inp, (N, H, W, C), torch.bfloat16)
    Ho, Wo = (H + 2 * pad - kh) // s + 1, (W + 2 * pad - kw) // s + 1
    K = kh * kw * C
    out = _tensor(registry, outp, (N * Ho * Wo, KP), torch.bfloat16)
    cols = F.unfold(x.permute(0, 3, 1, 2).float(), (kh, kw), padding=pad, stride=s)          # [N, C*kh*kw, L], (c, ky, kx)
    cols = cols.view(N, C, kh * kw, Ho * Wo).permute(0, 3, 2, 1).reshape(N * Ho * Wo, K)     # -> (ky, kx, c) columns
    ok = torch.equal(out[:, :K].view(torch.int16), cols.to(torch.bfloat16).view(torch.int16))
    return ok and bool((out[:, K:].view(torch.int16) == 0).all())


def _check_maxpool_call(registry, args):
    inp, outp, N, H, W, C = args[:6]
    x = _tensor(registry, inp, (N, H, W, C), torch.bfloat16)
    out = _tensor(registry, outp, (N, (H - 1) // 2 + 1, (W - 1) // 2 + 1, C), torch.bfloat16)
    want = F.max_pool2d(x.permute(0, 3, 1, 2).float(), 3, 2, 1).permute(0, 2, 3, 1)
    return torch.equal(out.float(), want)                # (value equality: fmaxf may pick either sign of a zero)


def _avgpool_ratio(x, out):
    """x [N, HW, C] bf16, out [N, C] fp32: worst |out - mean| / (HW 2^-24 mean|x| + 2^-24 |mean|) (sequential fp32 sum of HW
    terms, then one division); NaN counts as infinite."""
    HW = x.shape[1]
    xd = x.double()
    want = xd.mean(1)
    bound = HW * 2.0 ** -24 * xd.abs().mean(1) + 2.0 ** -24 * want.abs()
    err = (out.double() - want).abs()
    ratio = torch.where(err == 0, torch.zeros_like(err), err / bound)
    return float(ratio.masked_fill(torch.isnan(ratio), math.inf).max())


@pytest.fixture(scope="module")
def hmr_model():
    return psynth.build_synthetic_hmr(SEED, DEV)


@pytest.mark.gpu
@pytest.mark.parametrize("crops", [32, 3])
def test_every_native_call_of_the_extractor(hmr_model, crops, monkeypatch):
    """32 crops: the batch bench.py times (37 of the 53 GEMMs on 192-wide tiles, up to 22 tiles per persistent CTA).  3 crops:
    a ragged last m-tile on every layer (147 rows at layer 4)."""
    model = hmr_model
    x = torch.from_numpy(psynth.make_image_batch(SEED, crops)).to(DEV)
    xf, calls, registry, pk = _record_extractor(model, x, monkeypatch)
    counts = collections.Counter(name for name, _ in calls)
    assert counts == {"tp_nchw_to_nhwc_bf16": 1, "tp_im2col_nhwc_bf16": 20, "tp_gemm_bf16_tc": 53,
                      "tp_maxpool3x3s2_nhwc_bf16": 1, "tp_avgpool_nhwc_bf16": 1}, counts
    names = _wire(calls, pk, x, crops)

    bad, report = [], []
    for label, (name, args) in zip(names, calls):
        if name == "tp_nchw_to_nhwc_bf16":
            xp, yp, N, C, H, W, CP = args[:7]
            y = _tensor(registry, yp, (N, H, W, CP), torch.bfloat16)
            want = torch.zeros(N, H, W, CP, device=DEV, dtype=torch.bfloat16)
            want[..., :C] = x.permute(0, 2, 3, 1).to(torch.bfloat16)
            if not torch.equal(y.view(torch.int16), want.view(torch.int16)):
                bad.append(f"{label}: not bit-exact")
        elif name == "tp_im2col_nhwc_bf16":
            if not _check_im2col_call(registry, args):
                bad.append(f"{label}: not bit-exact against F.unfold")
        elif name == "tp_maxpool3x3s2_nhwc_bf16":
            if not _check_maxpool_call(registry, args):
                bad.append(f"{label}: not bit-exact against F.max_pool2d")
        elif name == "tp_avgpool_nhwc_bf16":
            inp, outp, N, HW, C = args[:5]
            out = _tensor(registry, outp, (N, C), torch.float32)
            assert out.data_ptr() == xf.data_ptr()
            ratio = _avgpool_ratio(_tensor(registry, inp, (N, HW, C), torch.bfloat16), out)
            report.append(f"{label:24s} ratio {ratio:.3f}")
            if not ratio <= 1.0:
                bad.append(f"{label}: avg-pool error ratio {ratio:.3g}")
        else:
            for r, (rows, cout), kp in _check_gemm_call(registry, args):
                bn = _tc_bn([(rows, cout)])
                tiles, per_cta = _tiles_per_cta([(rows, cout)], bn)
                tile = (r.row // TC_BM * TC_BM, r.col // bn * bn)
                report.append(f"{label:24s} rows {rows:6d} cout {cout:4d} kp {kp:4d}  BN {bn}  tiles {tiles:4d} "
                              f"(<= {per_cta:2d} per CTA)  worst ratio {r.ratio:.3f} at tile (m0, n0) = {tile}")
                if r.nans or not r.ratio <= 1.0:
                    bad.append(f"{label}: worst ratio {r.ratio:.3g} ({r.nans} NaN) at row {r.row} col {r.col}, "
                               f"tile (m0, n0) = {tile} of 128 x {bn}")
    print(f"\nHMR.feature_extractor, {crops} crops: every native call against float64 (ratio = |err| / bound)")
    print("\n".join(report))
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
def test_graphed_extractor_is_bit_identical_to_eager(hmr_model):
    """GraphedHMRFeatures(model, 32) is what bench.py times."""
    from tepose_b200.graph import GraphedHMRFeatures
    x = torch.from_numpy(psynth.make_image_batch(SEED, 32)).to(DEV)
    with torch.no_grad():
        eager = hmr_model.feature_extractor(x).clone()
    g = GraphedHMRFeatures(hmr_model, 32)
    got = g(x)
    torch.cuda.synchronize()
    assert g.launches_per_replay == 76
    assert torch.equal(got, eager)


# -------------------------------------------------------------------------------------------- standalone tp_gemm_bf16_tc
def _operands(rows, w_rows, kp, seed):
    g = torch.Generator(DEV).manual_seed(seed)
    A = torch.randn(rows, kp, generator=g, device=DEV).to(torch.bfloat16)
    W = (torch.randn(w_rows, kp, generator=g, device=DEV) / kp ** 0.5).to(torch.bfloat16)
    return A, W, g


class _Seg:
    """One segment with its own NaN-filled output buffer, larger than the segment: `extra` rows past m_rows, ldc > n_cols,
    and the output pointer `offset` elements into the buffer."""

    def __init__(self, g, m_start, m_rows, n_start, n_cols, *, relu=False, bf16=False, bias=True, residual=False,
                 ldc=None, offset=0, extra=3):
        from tepose_b200 import _native as nv
        self.m_start, self.m_rows, self.n_start, self.n_cols, self.relu = m_start, m_rows, n_start, n_cols, relu
        self.dtype = torch.bfloat16 if bf16 else torch.float32
        ldc = ldc or n_cols + 24
        self.buf = torch.full(((m_rows + extra) * ldc + offset,), float("nan"), device=DEV, dtype=self.dtype)
        self.bits0 = self.buf.view(INT_VIEW[self.dtype]).clone()
        self.inside = torch.zeros(self.buf.shape, device=DEV, dtype=torch.bool)
        self.inside[offset:offset + m_rows * ldc].view(m_rows, ldc)[:, :n_cols] = True
        self.out = self.buf[offset:offset + m_rows * ldc].view(m_rows, ldc)[:, :n_cols]
        self.bias = torch.randn(n_cols, generator=g, device=DEV) if bias else None
        ldr = n_cols + 8
        self.res_buf = torch.randn(m_rows, ldr, generator=g, device=DEV).to(torch.bfloat16) if residual else None
        self.residual = self.res_buf[:, :n_cols] if residual else None
        flags = (nv.GEMM_RELU if relu else 0) | (nv.GEMM_OUT_BF16 if bf16 else 0)
        self.seg = nv.GemmSeg(m_start, m_rows, n_start, n_cols, nv.vp(self.buf.data_ptr() + offset * self.buf.element_size()), ldc,
                              nv.ptr(self.bias), flags, ldr if residual else 0, nv.ptr(self.res_buf))


def _launch(A, W, segs):
    from tepose_b200 import _native as nv
    arr = (nv.GemmSeg * len(segs))(*[s.seg for s in segs])
    rc = nv.lib().tp_gemm_bf16_tc(nv.ptr(A), A.shape[0], nv.ptr(W), W.shape[0], A.shape[1], arr, len(segs), nv.stream())
    torch.cuda.synchronize()
    return rc


def _run_and_check(A, W, segs):
    from tepose_b200 import _native as nv
    nv.check(_launch(A, W, segs), "tp_gemm_bf16_tc")
    bn = _tc_bn([(s.m_rows, s.n_cols) for s in segs])
    for i, s in enumerate(segs):
        r = gemm_check(A[s.m_start:s.m_start + s.m_rows], W[s.n_start:s.n_start + s.n_cols], s.bias, s.residual, s.relu, s.out)
        tile = (r.row // TC_BM * TC_BM, r.col // bn * bn)
        assert r.nans == 0 and r.ratio <= 1.0, f"segment {i}: worst ratio {r.ratio:.3g} ({r.nans} NaN), tile (m0, n0) = {tile}, BN {bn}"
        changed = (s.buf.view(INT_VIEW[s.dtype]) != s.bits0) & ~s.inside
        assert not bool(changed.any()), f"segment {i}: {int(changed.sum())} elements written outside the segment"
    return bn


MANY_ROWS, MANY_COLS = 1000, 25008     # 8 m-tiles (last one 104 rows) x 131 n-tiles of 192 (last one 48 columns) = 1048 tiles


@pytest.mark.gpu
@pytest.mark.parametrize("kp", [64, 4096])
@pytest.mark.parametrize("relu,bf16,residual", list(itertools.product([False, True], repeat=3)))
def test_gemm_many_tiles_per_cta(kp, relu, bf16, residual):
    """1048 tiles on 148 persistent CTAs: 8 tiles on the first CTAs, consecutive tiles of a CTA 18.5 n-tiles apart, so every
    tile brings a new bias into s_bias[acc] and both TMEM accumulators cycle several times.  kp = 64: one k-block per tile (the
    accumulate = 0 first step on every tile); kp = 4096: the smem ring wraps many times within each tile."""
    A, W, g = _operands(MANY_ROWS, MANY_COLS + 48, kp, kp + 8 * relu + 4 * bf16 + 2 * residual)
    s = _Seg(g, 0, MANY_ROWS, 16, MANY_COLS, relu=relu, bf16=bf16, residual=residual)
    bn = _run_and_check(A, W, [s])
    assert bn == 192 and _tiles_per_cta([(MANY_ROWS, MANY_COLS)], bn)[1] >= 8


@pytest.mark.gpu
@pytest.mark.parametrize("ldc_extra,offset,relu,residual", [(3, 0, False, False), (8, 1, True, True)])
def test_gemm_fp32_output_without_vector_stores(ldc_extra, offset, relu, residual):
    """fp32 output with ldc % 4 != 0, or with the output pointer 4 bytes past a 16-byte boundary: the scalar store path."""
    A, W, g = _operands(MANY_ROWS, MANY_COLS, 64, 11 + offset)
    s = _Seg(g, 0, MANY_ROWS, 0, MANY_COLS, relu=relu, residual=residual, ldc=MANY_COLS + ldc_extra, offset=offset)
    assert (s.seg.out % 16 != 0) == (offset != 0)
    _run_and_check(A, W, [s])


@pytest.mark.gpu
@pytest.mark.parametrize("past_one_wave", [0, 1])
def test_gemm_tile_width_switch(past_one_wave):
    """tiles128 == SM count keeps 128-wide tiles; one more switches to 192, where the only n-tile holds 128 of its 192 columns."""
    sm = torch.cuda.get_device_properties(DEV).multi_processor_count
    rows = (sm + past_one_wave) * TC_BM - 40
    A, W, g = _operands(rows, 320, 256, 21 + past_one_wave)
    for bf16, residual in ((False, False), (True, True)):
        s = _Seg(g, 0, rows, 64, 128, relu=bf16, bf16=bf16, residual=residual)
        assert _run_and_check(A, W, [s]) == (192 if past_one_wave else 128)


@pytest.mark.gpu
def test_gemm_eight_segments():
    """TC_MAX_SEGS segments, each with its own rows, columns, output, flags and residual (one without bias): every slot of
    tc_decode's static select, a single-row segment and an odd n_start."""
    A, W, g = _operands(1500, 1200, 192, 31)
    spec = [(0, 300, 0, 160, dict(relu=True, bf16=True, residual=True)),
            (37, 129, 160, 64, dict(bf16=True)),
            (200, 1, 304, 16, dict(relu=True)),
            (511, 400, 96, 336, dict(residual=True)),
            (1000, 500, 640, 560, dict(relu=True, bf16=True)),
            (5, 128, 1184, 16, dict(bias=False, residual=True, bf16=True)),
            (777, 255, 17, 48, dict(relu=True, residual=True)),
            (1400, 100, 400, 48, dict(bf16=True, residual=True))]
    segs = [_Seg(g, m0, mr, n0, nc, **kw) for m0, mr, n0, nc, kw in spec]
    _run_and_check(A, W, segs)


@pytest.mark.gpu
def test_gemm_rejects_n_cols_not_a_multiple_of_16():
    from tepose_b200 import _native as nv
    A, W, g = _operands(128, 64, 64, 41)
    s = _Seg(g, 0, 128, 0, 40)
    assert _launch(A, W, [s]) == -1                                   # TP_ERR_INVALID
    assert b"n_cols" in nv.lib().tp_last_error()
    assert bool(torch.isnan(s.buf).all())


# -------------------------------------------------------------------------------------- pooling and layout kernels
def _guarded(n, dtype):
    """A NaN buffer of n elements plus a 64-element tail that must stay NaN."""
    buf = torch.full((n + 64,), float("nan"), device=DEV, dtype=dtype)
    return buf, buf[:n]


@pytest.mark.gpu
@pytest.mark.parametrize("size", [112, 113])
def test_maxpool_production_shape(size):
    """[32,112,112,64] is the stem's max-pool at 32 crops; 113 x 113 has a last window that hangs over the bottom/right edge.
    All inputs are negative, so a border window that took the padding as 0 would show."""
    from tepose_b200 import _native as nv
    g = torch.Generator(DEV).manual_seed(size)
    x = (-(torch.rand(32, size, size, 64, generator=g, device=DEV) * 4 + 0.01)).to(torch.bfloat16)
    Ho = (size - 1) // 2 + 1
    buf, out = _guarded(32 * Ho * Ho * 64, torch.bfloat16)
    nv.check(nv.lib().tp_maxpool3x3s2_nhwc_bf16(nv.ptr(x), nv.ptr(out), 32, size, size, 64, nv.stream()))
    want = F.max_pool2d(x.permute(0, 3, 1, 2).float(), 3, 2, 1).permute(0, 2, 3, 1).to(torch.bfloat16).contiguous()
    assert torch.equal(out.view(torch.int16), want.view(-1).view(torch.int16))
    assert bool(torch.isnan(buf[out.numel():]).all())


@pytest.mark.gpu
def test_avgpool_production_shape():
    from tepose_b200 import _native as nv
    g = torch.Generator(DEV).manual_seed(49)
    x = (torch.randn(32, 49, 2048, generator=g, device=DEV) + 0.5).to(torch.bfloat16)
    buf, out = _guarded(32 * 2048, torch.float32)
    nv.check(nv.lib().tp_avgpool_nhwc_bf16(nv.ptr(x), nv.ptr(out), 32, 49, 2048, nv.stream()))
    torch.cuda.synchronize()
    assert _avgpool_ratio(x, out.view(32, 2048)) <= 1.0
    assert bool(torch.isnan(buf[out.numel():]).all())


@pytest.mark.gpu
def test_nchw_to_nhwc_production_shape():
    from tepose_b200 import _native as nv
    g = torch.Generator(DEV).manual_seed(3)
    x = torch.randn(32, 3, 224, 224, generator=g, device=DEV) * 3
    buf, out = _guarded(32 * 224 * 224 * 4, torch.bfloat16)
    nv.check(nv.lib().tp_nchw_to_nhwc_bf16(nv.ptr(x), nv.ptr(out), 32, 3, 224, 224, 4, nv.stream()))
    want = torch.zeros(32, 224, 224, 4, device=DEV, dtype=torch.bfloat16)
    want[..., :3] = x.permute(0, 2, 3, 1).to(torch.bfloat16)
    assert torch.equal(out.view(torch.int16), want.view(-1).view(torch.int16))
    assert bool(torch.isnan(buf[out.numel():]).all())
