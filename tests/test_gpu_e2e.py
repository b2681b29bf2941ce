"""GPU end-to-end parity: tepose_b200.TePose (CUDA kernels through the C ABI) against the
golden vectors produced by the unmodified reference and against the CPU oracle."""
import os

import pytest
import torch

from oracle import synth, torch_ref
from tests.helpers import build_product_model, compare_outputs, load_forward_golden, oracle_forward

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
DEV = "cuda:0"


@pytest.mark.parametrize("fname", sorted(f for f in os.listdir(GOLD) if f.startswith("fwd_")))
@pytest.mark.parametrize("precision", ["fp32", "bf16", "fp32_tc"])
def test_forward_against_reference_golden(fname, precision):
    cfg, gold, cut = load_forward_golden(os.path.join(GOLD, fname))
    model, sd = build_product_model(cfg["seed"], cfg["seqlen"], cfg["n_layers"], cfg["hidden"], precision, DEV)
    x = torch.from_numpy(synth.make_input(cfg["seed"], cfg["batch"], cfg["seqlen"])).to(DEV)
    Jr = torch_ref.SmplModel.synthetic(cfg["seed"]).J_regressor_h36m.to(DEV) if cfg.get("use_h36m") else None
    out = cut(model(x, is_train=cfg.get("is_train", False), J_regressor=Jr)[-1])
    if precision in ("fp32", "fp32_tc"):   # north_star: <= 1e-4 m on verts / joints in fp32 (fp32_tc: K1 / K2 as 3-term bf16 splits on tensor cores)
        errs = compare_outputs(out, gold, label=fname)
    else:                     # north_star: <= 1 mm in bf16
        errs = compare_outputs(out, gold, vert_tol=1e-3, rot_tol=2e-3, kp2d_tol=5e-2, label=fname)
    print(fname, precision, errs)


@pytest.mark.parametrize("precision", ["fp32", "bf16", "fp32_tc"])
@pytest.mark.parametrize("L,H,T,B", [(1, 2048, 16, 32), (2, 1024, 6, 32), (1, 2048, 16, 1)])
def test_forward_full_size_against_oracle(L, H, T, B, precision):
    """BASELINE configs at full size (defaults L=1,H=2048,T=16; released L=2,H=1024,T=6)."""
    seed = 40 + L
    model, sd = build_product_model(seed, T, L, H, precision, DEV)
    x = synth.make_input(seed, B, T)
    ref, m = oracle_forward(seed, sd, x, L, H)
    out = model(torch.from_numpy(x).to(DEV))[-1]
    if precision in ("fp32", "fp32_tc"):
        errs = compare_outputs(out, ref, label=f"L{L}H{H}")
    else:
        errs = compare_outputs(out, ref, vert_tol=1e-3, rot_tol=2e-3, kp2d_tol=5e-2, label=f"L{L}H{H}")
        mpjpe = float((out["kp_3d"].cpu() - ref["kp_3d"]).norm(dim=-1).mean())
        assert mpjpe < 1e-3, mpjpe        # <= 1 mm MPJPE delta
    print(L, H, T, B, precision, errs)


@pytest.mark.parametrize("precision,H,graph", [("fp32", 256, False), ("bf16", 2048, True)])
def test_live_stream_carried_state(precision, H, graph):
    """Config 3: causal carried-state stepping (B=1) against torch.nn.GRU stepped with explicit h0."""
    from tepose_b200.live import LiveTePose
    seed, B, N = 51, 1, 6
    model, sd = build_product_model(seed, 16, 1, H, precision, DEV)
    m = torch_ref.SmplModel.synthetic(seed)
    feats = torch.from_numpy(synth.make_input(seed, B, N))[:, :, :2048]
    live = LiveTePose(model, batch=B, use_graph=graph)
    outs = [{k: v.clone().cpu() for k, v in live.step(feats[:, t].to(DEV)).items()} for t in range(N)]
    hF = hB = prev = None
    tol = {} if precision == "fp32" else dict(vert_tol=1e-3, rot_tol=2e-3, kp2d_tol=5e-2)
    for t in range(N):
        newest = torch.cat([feats[:, t], torch.zeros(B, 85)], dim=1)[:, None]
        if prev is None:
            hFt, hBt, hS = torch_ref.encoder_causal_states(sd, newest, H)
        else:
            hF, hB, _ = torch_ref.encoder_causal_states(sd, prev, H, h0=None if hF is None else (hF, hB))
            hFt, hBt, hS = torch_ref.encoder_causal_states(sd, newest, H, h0=(hF, hB))
        ref = torch_ref.regressor_forward(sd, m, torch_ref.encoder_from_states(sd, hFt, hBt, hS))
        compare_outputs(outs[t], ref, label=f"live {precision} frame {t}", **tol)
        # feed the oracle its own theta (the product feeds back its own): both chains stay within tolerance
        prev = torch.cat([feats[:, t], ref["theta"]], dim=1)[:, None]


def test_graphed_forward_equals_eager():
    from tepose_b200.graph import GraphedTePose
    model, sd = build_product_model(61, 16, 1, 256, "bf16", DEV)
    x = torch.from_numpy(synth.make_input(61, 4, 16)).to(DEV)
    eager = {k: v.clone() for k, v in model(x)[-1].items()}
    g = GraphedTePose(model, 4, 16)
    out = g(x)
    torch.cuda.synchronize()
    for k in eager:
        assert torch.equal(out[k], eager[k]), k          # same kernels, same order: bitwise
    assert g.launches_per_replay >= 6


def test_pipelined_host_buffer_api_matches_direct_forward():
    """tepose_b200.pipeline: overlapped H2D / compute / D2H must return exactly the direct results."""
    from tepose_b200.pipeline import PipelinedTePose
    model, sd = build_product_model(71, 16, 1, 256, "bf16", DEV)
    xs = [torch.from_numpy(synth.make_input(71 + i, 4, 16)).pin_memory() for i in range(7)]
    direct = [{k: v.clone().cpu() for k, v in model(x.to(DEV))[-1].items()} for x in xs]
    pipe = PipelinedTePose(model, 4, 16, depth=3)
    tickets, got = [], []
    for x in xs:
        tickets.append(pipe.submit(x))
        if len(tickets) >= pipe.depth:
            got.append({k: v.clone() for k, v in pipe.result(tickets.pop(0)).items()})
    for tk in tickets:
        got.append({k: v.clone() for k, v in pipe.result(tk).items()})
    assert len(got) == len(xs)
    for a, b in zip(got, direct):
        for k in a:
            assert torch.equal(a[k], b[k]), k
    with pytest.raises(ValueError):
        pipe.result(0)          # slot already recycled


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("L,H,T,B,train,h36m", [
    (1, 256, 1, 3, False, False),      # single-frame window
    (1, 256, 16, 33, False, True),     # batch just above one MMA tile -> generic recurrence path, H36M joints
    (1, 128, 5, 64, False, False),     # 64 sequences
    (2, 256, 6, 32, True, False),      # released depth, train-shaped output (2 rows per sequence)
    (3, 96, 4, 2, False, False),       # three layers, H not a multiple of 128
    (1, 2048, 16, 7, False, False),    # ragged batch at full width
    (1, 128, 4, 80, False, False),     # more rows than one 64-row chunk of the skinny kernels
    (1, 128, 3, 40, True, True),       # train-shaped: 80 regressor rows from 40 sequences
])
def test_forward_edge_shapes_against_oracle(L, H, T, B, train, h36m, precision):
    seed = 80 + L + B
    model, sd = build_product_model(seed, T, L, H, precision, DEV)
    x = synth.make_input(seed, B, T)
    ref, m = oracle_forward(seed, sd, x, L, H, is_train=train, use_h36m=h36m)
    Jr = m.J_regressor_h36m.to(DEV) if h36m else None
    out = model(torch.from_numpy(x).to(DEV), is_train=train, J_regressor=Jr)[-1]
    tol = {} if precision == "fp32" else dict(vert_tol=1e-3, rot_tol=2e-3, kp2d_tol=5e-2)
    compare_outputs(out, ref, label=f"L{L}H{H}T{T}B{B}", **tol)


def test_non_contiguous_and_repeated_calls():
    """Inputs that are views (strided batch / time) and back-to-back calls must give identical results."""
    model, sd = build_product_model(90, 8, 1, 256, "fp32", DEV)
    big = torch.from_numpy(synth.make_input(90, 6, 16)).to(DEV)
    view = big[::2, 4:12]                       # non-contiguous in batch and time
    a = model(view)[-1]
    b = model(view.contiguous())[-1]
    c = model(view)[-1]
    for k in a:
        assert torch.equal(a[k], b[k]) and torch.equal(a[k], c[k]), k


def test_errors_are_loud():
    model, _ = build_product_model(91, 4, 1, 128, "fp32", DEV)
    with pytest.raises(ValueError):
        model(torch.zeros(2, 4, 100, device=DEV))              # wrong feature width
    with pytest.raises(RuntimeError):
        model(torch.zeros(2, 4, 2133))                          # CPU tensor: no fallback
    model.train()
    with pytest.raises(NotImplementedError):
        model(torch.zeros(2, 4, 2133, device=DEV))


# ------------------------------------------------------------------------------------------------ folded heads + IEF
@pytest.mark.parametrize("fname", sorted(f for f in os.listdir(GOLD) if f.startswith("fwd_") and "train" not in f))
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_folded_forward_against_reference_golden(fname, precision):
    """fold_linear=True: heads + IEF as one pre-composed affine map (TePose.folded) -- same tolerances."""
    cfg, gold, cut = load_forward_golden(os.path.join(GOLD, fname))
    model, sd = build_product_model(cfg["seed"], cfg["seqlen"], cfg["n_layers"], cfg["hidden"], precision, DEV)
    model.fold_linear = True
    x = torch.from_numpy(synth.make_input(cfg["seed"], cfg["batch"], cfg["seqlen"])).to(DEV)
    Jr = torch_ref.SmplModel.synthetic(cfg["seed"]).J_regressor_h36m.to(DEV) if cfg.get("use_h36m") else None
    out = cut(model(x, J_regressor=Jr)[-1])
    tol = {} if precision == "fp32" else dict(vert_tol=1e-3, rot_tol=2e-3, kp2d_tol=5e-2)
    print(fname, precision, compare_outputs(out, gold, label=fname, **tol))


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_folded_forward_full_size(precision):
    from tepose_b200.graph import GraphedTePose
    seed, L, H, T, B = 47, 1, 2048, 16, 32
    model, sd = build_product_model(seed, T, L, H, precision, DEV)
    x = synth.make_input(seed, B, T)
    ref, m = oracle_forward(seed, sd, x, L, H)
    xd = torch.from_numpy(x).to(DEV)
    plain = {k: v.clone() for k, v in model(xd)[-1].items()}
    model.fold_linear = True
    out = model(xd)[-1]
    tol = {} if precision == "fp32" else dict(vert_tol=1e-3, rot_tol=2e-3, kp2d_tol=5e-2)
    errs = compare_outputs(out, ref, label="folded full", **tol)
    e_plain = compare_outputs(plain, ref, label="plain full", **tol)
    print(precision, "folded", errs, "layer-by-layer", e_plain)
    g = GraphedTePose(model, B, T)
    rep = g(xd)
    for k in out:
        assert torch.equal(rep[k], out[k]), k
    assert g.launches_per_replay < 12


# ------------------------------------------------------------------------------------------------ launch structure
@pytest.mark.parametrize("B,T,L,H", [(32, 16, 1, 2048), (1, 16, 1, 2048), (32, 6, 2, 1024)])
def test_programmatic_dependent_launch_does_not_change_results(B, T, L, H):
    """Every kernel of a forward is PDL-linked to its predecessor (set-up overlaps the predecessor's tail, then
    griddepcontrol.wait).  A kernel that touched its inputs before the wait would race: results with the overlap on
    (eager and graph replay, repeated) must be bit-identical to the fully serialised run."""
    from tepose_b200 import _native as nv
    from tepose_b200.graph import GraphedTePose
    model, _ = build_product_model(95, T, L, H, "bf16", DEV)
    x = torch.from_numpy(synth.make_input(95, B, T)).to(DEV)
    was = nv.lib().tp_set_pdl(0)
    try:
        ref = {k: v.clone() for k, v in model(x)[-1].items()}
    finally:
        nv.lib().tp_set_pdl(1)
    assert was == 1
    g = GraphedTePose(model, B, T)
    for rep in range(5):
        out = model(x)[-1]
        for k in ref:
            assert torch.equal(out[k], ref[k]), ("eager", rep, k)
        out = g(x)
        for k in ref:
            assert torch.equal(out[k], ref[k]), ("graph", rep, k)


def test_fused_heads_ief_kernel_against_separate_kernels():
    """tp_heads_ief_forward (heads as leading layers of the persistent IEF kernel) vs tp_encoder_heads_cat + tp_ief_forward."""
    model, _ = build_product_model(96, 16, 1, 2048, "bf16", DEV)
    x = torch.from_numpy(synth.make_input(96, 32, 16)).to(DEV)
    fused = {k: v.clone() for k, v in model(x)[-1].items()}
    model.fuse_heads = False
    try:
        sep = model(x)[-1]
    finally:
        model.fuse_heads = True
    # same bf16 operands, fp32 accumulation in a different order (K slices / split-K)
    assert float((fused["theta"] - sep["theta"]).abs().max()) < 2e-4
    assert float((fused["verts"] - sep["verts"]).abs().max()) < 1e-4


@pytest.mark.gpu
def test_forward_on_a_non_current_device():
    """A model and input on cuda:1 while cuda:0 is the current device (ADVICE r1): the entry points switch the current device
    themselves, the outputs live on cuda:1 and match the same forward run with cuda:1 current."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from tepose_b200 import synthetic as psynth
    x = torch.from_numpy(psynth.make_input(3, 4, 8))
    torch.cuda.set_device(1)
    model, _ = psynth.build_synthetic_model(3, 8, 1, 256, "bf16", "cuda:1")
    with torch.no_grad():
        want = model(x.to("cuda:1"))[-1]
    torch.cuda.set_device(0)
    with torch.no_grad():
        got = model(x.to("cuda:1"))[-1]
    torch.cuda.synchronize("cuda:1")
    for k in want:
        assert got[k].device == want[k].device == torch.device("cuda:1")
        assert torch.equal(got[k], want[k]), k


def test_pipeline_float16_rows_and_output_selection():
    """PipelinedTePose(outputs=..., input_dtype=torch.float16): the float16 rows are widened by the pack kernel (bit-identical to
    feeding the same values as float32), only the requested outputs reach the host, and they equal the full pipeline's."""
    from tepose_b200.pipeline import PipelinedTePose
    from tepose_b200 import synthetic as psynth
    B, T = 5, 8
    model, _ = psynth.build_synthetic_model(7, T, 1, 256, "bf16", DEV)
    x16 = torch.from_numpy(psynth.make_input(7, B, T)).to(torch.float16)
    x32 = x16.float()
    full = PipelinedTePose(model, B, T, depth=2)
    lean = PipelinedTePose(model, B, T, depth=2, outputs=("theta", "kp_3d", "rotmat"), input_dtype=torch.float16)
    assert lean.h2d_bytes * 2 == full.h2d_bytes and lean.d2h_bytes < full.d2h_bytes // 20
    with torch.no_grad():
        a = {k: v.clone() for k, v in full.result(full.submit(x32.pin_memory())).items()}
        b = {k: v.clone() for k, v in lean.result(lean.submit(x16.pin_memory())).items()}
        direct = model(x16.to(DEV))[-1]
    assert set(b) == {"theta", "kp_3d", "rotmat"}
    for k in b:
        assert torch.equal(a[k], b[k]), k
        assert torch.equal(direct[k].cpu().reshape(b[k].shape), b[k]), k


def test_acquire_fence_build_is_bit_identical():
    """VERDICT r1 / ADVICE r1: the grid barriers of the persistent kernels poll with relaxed loads and skip the formal acquire fence
    (every post-barrier read of another CTA's data is an L2-coherent access).  The same sources built with -DTP_BARRIER_ACQUIRE_FENCE
    (tepose_b200/build.py variant 'fence') must give bit-identical outputs at the headline shape, with and without CUDA graph + PDL."""
    import hashlib
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    fence = os.path.join(root, "tepose_b200", "libtepose_b200_fence.so")
    if not os.path.isfile(fence):
        pytest.skip("libtepose_b200_fence.so not built (python -m tepose_b200.build --fence)")
    prog = (
        "import sys, hashlib, torch; sys.path.insert(0, %r)\n"
        "from tepose_b200 import synthetic as s\n"
        "from tepose_b200.graph import GraphedTePose\n"
        "import tepose_b200._native as nv\n"
        "h = hashlib.sha256()\n"
        "for prec, B, T, L, H in (('bf16', 32, 16, 1, 2048), ('bf16', 5, 6, 2, 256), ('fp32', 4, 8, 1, 128)):\n"
        "    m, _ = s.build_synthetic_model(3, T, L, H, prec, 'cuda:0')\n"
        "    x = torch.from_numpy(s.make_input(3, B, T)).cuda()\n"
        "    with torch.no_grad():\n"
        "        o = m(x)[-1]\n"
        "        g = GraphedTePose(m, B, T); g.static_input.copy_(x); og = g.replay()\n"
        "    torch.cuda.synchronize()\n"
        "    for k in sorted(o):\n"
        "        assert torch.equal(o[k], og[k].reshape(o[k].shape)), k\n"
        "        h.update(o[k].cpu().numpy().tobytes())\n"
        "print('DIGEST', h.hexdigest(), nv.LIB_PATH)\n") % root
    digests = []
    for lib in (None, fence):
        env = dict(os.environ)
        env.pop("TEPOSE_B200_LIB", None)
        if lib:
            env["TEPOSE_B200_LIB"] = lib
        r = subprocess.run([sys.executable, "-c", prog], env=env, capture_output=True, text=True, timeout=900, cwd=root)
        assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
        line = [ln for ln in r.stdout.splitlines() if ln.startswith("DIGEST")][-1].split()
        assert (lib or "libtepose_b200.so") in line[2]
        digests.append(line[1])
    assert digests[0] == digests[1], digests
