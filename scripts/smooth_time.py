"""Times the pose smoothing (tepose_b200.smooth) on cuda:0 and prints one JSON line:

- smooth_pose for one 1000-frame track (one filter launch + one SMPL call over the 1000 rows): CUDA events around each call,
  median of --reps calls; the filter launch alone the same way;
- the added cost per push of TrackedTePose(smooth=(0.004, 0.7)) at S = 8 in the released configuration (T6 L2 H1024, seeded
  tracks, every slot present), bf16 and fp32: smooth=None and smooth=(0.004, 0.7) timed in alternation, --rounds rounds of
  --pushes back-to-back steady pushes each, one synchronize per round; the median round is reported per push;
- for context, the reference's pattern on the first frames of that track: the numpy float32 filter, then SMPL once per frame at batch 1
  on the CPU (oracle.torch_ref), host clock over --reference-frames frames.

Synthetic weights.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import smooth_ref, synth, torch_ref  # noqa: E402
from scripts.video_time import card  # noqa: E402
from tepose_b200 import TrackedTePose, smooth_pose  # noqa: E402
from tepose_b200.smooth import one_euro_filter  # noqa: E402
from tepose_b200.stream import FEAT  # noqa: E402
from tepose_b200.synthetic import build_synthetic_model  # noqa: E402

DEV = "cuda:0"
N = 1000
PARAMS = (0.004, 0.7)


def events_ms(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return {"ms_median": round(float(np.median(times)), 4), "ms_min": round(float(min(times)), 4)}


def track(seed, n):
    b = synth.make_bodies(seed, n)
    pose = b["pose_aa"].astype(np.float32) + np.cumsum(0.01 * np.random.default_rng(seed).standard_normal((n, 72)), 0).astype(np.float32)
    return pose, b["betas"].astype(np.float32)


def push_cost(precision, S, pushes, rounds):
    T, L, H = 6, 2, 1024
    model, _ = build_synthetic_model(0, T, L, H, precision, DEV)
    g = torch.Generator().manual_seed(1)
    feats = torch.randn(64, S, FEAT, generator=g).to(DEV)
    seeds = {i: 0.1 * torch.randn(T - 1, 85, generator=g) for i in range(S)}
    ids = list(range(S))
    trackers = {"off": TrackedTePose(model, None, slots=S), "on": TrackedTePose(model, None, slots=S, smooth=PARAMS)}
    for tt in trackers.values():                     # start every track, pass the T-th push, warm the graphs
        for k in range(T + 10):
            tt.push(feats[k % 64], ids, theta_input=seeds if k == 0 else None)
    torch.cuda.synchronize()
    per = {"off": [], "on": []}
    for r in range(rounds):
        for name, tt in trackers.items():
            t0 = time.perf_counter()
            for k in range(pushes):
                tt.push(feats[k % 64], ids)
            torch.cuda.synchronize()
            per[name].append((time.perf_counter() - t0) / pushes * 1e3)
    off, on = float(np.median(per["off"])), float(np.median(per["on"]))
    return {"push_ms_smooth_off": round(off, 4), "push_ms_smooth_on": round(on, 4), "added_ms": round(on - off, 4),
            "rounds_off_ms": [round(v, 4) for v in per["off"]], "rounds_on_ms": [round(v, 4) for v in per["on"]],
            "launches_per_replay_off": trackers["off"].launches_per_replay,
            "launches_per_replay_on": trackers["on"].launches_per_replay}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--pushes", type=int, default=100, help="pushes per timed round")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reference-frames", type=int, default=200, help="frames of the CPU reference pattern (its time per frame is reported)")
    args = ap.parse_args()
    torch.cuda.init()
    res = {"card": card(), "model": "synthetic weights; TePose T6 L2 H1024 (released configuration), seeded tracks"}

    model, _ = build_synthetic_model(0, 6, 2, 1024, "fp32", DEV)
    smpl = model.regressor.smpl
    pose, betas = track(3, N)
    pd, bd = torch.from_numpy(pose).to(DEV), torch.from_numpy(betas).to(DEV)
    res["smooth_pose_1000"] = events_ms(lambda: smooth_pose(pd, bd, *PARAMS, smpl=smpl), args.reps)
    out, state = torch.empty(1, N, 72, device=DEV), torch.empty(1, 2, 72, device=DEV)
    table = torch.tensor([N, 1], dtype=torch.int32, device=DEV)
    res["filter_1000"] = events_ms(lambda: one_euro_filter(pd.view(1, N, 72), out, state, table[0:1], table[1:2], N, *PARAMS),
                                   args.reps)
    del model

    res["push_S8"] = {p: push_cost(p, 8, args.pushes, args.rounds) for p in ("bf16", "fp32")}

    m = torch_ref.SmplModel.synthetic(0)
    n = args.reference_frames
    t0 = time.perf_counter()
    smooth_ref.smooth_pose(m, pose[:n], betas[:n], *PARAMS)
    dt = time.perf_counter() - t0
    res["reference_cpu"] = {"frames": n, "s": round(dt, 3), "ms_per_frame": round(dt / n * 1e3, 3),
                            "torch_threads": torch.get_num_threads()}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
