"""Times the per-track video path (tepose_b200.TrackedVideoTePose) on cuda:0 and prints one JSON line:

- frames per second at 1, 4, 16 and 32 people present with slots = 32, next to VideoTePose(batch=32) on the same boxes (the
  P boxes repeated up to 32 rows: what a fixed batch of 32 pays for P people).  The two are timed in alternation, --rounds
  rounds of --pushes back-to-back pushes each, one synchronize per round; the median round is reported;
- push latency at slots = 8 with one person present: host clock around push() + synchronize, p50 / p99;
- the two slot kernels alone at S = 32, T = 16 (every slot op 1): CUDA events around a graph of 20 launches.

The configuration of scripts/video_time.py: 1920x1080 RGB frames already on the device, HMR and TePose T16 L1 H2048 bf16, VIBE
L2 H1024 bf16, synthetic weights.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import crop_ref  # noqa: E402
from scripts.video_time import H, W, T, boxes, card  # noqa: E402
from tepose_b200 import TrackedVideoTePose, VideoTePose, _native as nv  # noqa: E402
from tepose_b200.stream import FEAT  # noqa: E402
from tepose_b200.synthetic import build_synthetic_hmr, build_synthetic_model, build_synthetic_vibe  # noqa: E402


def tracked_push(tv, frames, P, i):
    tv.push(frames[i % len(frames)], {p: tuple(r) for p, r in enumerate(boxes(P, i))})


def fixed_push(vt, frames, P, i):
    rows = boxes(P, i)
    vt.push(frames[i % len(frames)], rows[np.arange(32) % P])


def timed(fn, n, start):
    t0 = time.perf_counter()
    for i in range(start, start + n):
        fn(i)
    torch.cuda.synchronize()
    return n / (time.perf_counter() - t0)


def kernel_us(S=32, T=T, reps=20):
    """The slot push and commit kernels alone, each in a graph of `reps` launches, CUDA events; median of 20 replays."""
    ld = FEAT + 85
    x = torch.randn(S, T, ld, device="cuda:0")
    feats = torch.randn(S, FEAT, device="cuda:0")
    theta = torch.randn(S, 85, device="cuda:0")
    tab = torch.stack([torch.ones(S, dtype=torch.int32), torch.arange(S, dtype=torch.int32)]).cuda()
    L = nv.lib()
    calls = {
        "push": lambda: nv.check(L.tp_window_slots_push(nv.ptr(x), S, T, ld, nv.ptr(feats), nv.ptr(tab[1]), nv.ptr(tab[0]),
                                                        nv.stream())),
        "commit": lambda: nv.check(L.tp_window_slots_commit(nv.ptr(x), S, T, ld, nv.ptr(theta), nv.ptr(tab[0]), nv.stream())),
    }
    out = {}
    for name, call in calls.items():
        call()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(reps):
                call()
        for _ in range(3):
            g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        times = []
        for _ in range(20):
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / reps * 1e3)
        out[name] = {"us_median": round(float(np.median(times)), 3), "us_min": round(float(min(times)), 3)}
    # bytes a launch moves at S = 32 (every slot op 1): push reads T-1 feature rows + 1 feats row and writes T per slot
    out["push"]["bytes"] = S * (2 * T) * FEAT * 4
    out["commit"]["bytes"] = S * (2 * (T - 1)) * 85 * 4
    out["S"], out["T"] = S, T
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pushes", type=int, default=100, help="pushes per timed round")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--latency-pushes", type=int, default=300)
    ap.add_argument("--clip", type=int, default=8, help="distinct frames cycled through")
    args = ap.parse_args()
    torch.cuda.init()
    dev = "cuda:0"
    hmr = build_synthetic_hmr(0, dev)
    model, _ = build_synthetic_model(0, T, 1, 2048, "bf16", dev)
    vibe, _ = build_synthetic_vibe(0, T, 2, 1024, True, False, True, "bf16", dev)
    host = torch.from_numpy(crop_ref.sample_frames(1, args.clip, H, W))
    frames = [host[i:i + 1].to(dev) for i in range(args.clip)]
    res = {"card": card(), "frame": [H, W],
           "model": "HMR bf16, TePose T16 L1 H2048 bf16, VIBE L2 H1024 bf16, synthetic weights",
           "method": f"median of {args.rounds} alternating rounds of {args.pushes} back-to-back pushes, device frames"}

    fps = {}
    for P in (1, 4, 16, 32):
        tv = TrackedVideoTePose(hmr, model, vibe, slots=32)
        vt = VideoTePose(hmr, model, vibe, batch=32)
        warm = T + 10
        timed(lambda i: tracked_push(tv, frames, P, i), warm, 0)             # bootstraps every track, captures, warms up
        timed(lambda i: fixed_push(vt, frames, P, i), warm, 0)
        a, b = [], []
        for r in range(args.rounds):
            start = warm + r * args.pushes
            a.append(timed(lambda i: tracked_push(tv, frames, P, i), args.pushes, start))
            b.append(timed(lambda i: fixed_push(vt, frames, P, i), args.pushes, start))
        fa, fb = float(np.median(a)), float(np.median(b))
        fps[f"P{P}"] = {"tracked_slots32_fps": round(fa, 1), "video_batch32_fps": round(fb, 1),
                        "tracked_over_video": round(fa / fb, 3), "trunk_batch": max(tv.buckets),
                        "tracked_rounds_fps": [round(v, 1) for v in a], "video_rounds_fps": [round(v, 1) for v in b]}
        del tv, vt
        torch.cuda.empty_cache()
    res["frames_per_s"] = fps

    tv = TrackedVideoTePose(hmr, model, vibe, slots=8)
    for i in range(T + 20):
        tracked_push(tv, frames, 1, i)
    torch.cuda.synchronize()
    lat = []
    for i in range(T + 20, T + 20 + args.latency_pushes):
        s = time.perf_counter()
        tracked_push(tv, frames, 1, i)
        torch.cuda.synchronize()
        lat.append(time.perf_counter() - s)
    ms = np.array(lat) * 1e3
    res["push_slots8_P1_ms"] = {"p50": round(float(np.percentile(ms, 50)), 4), "p99": round(float(np.percentile(ms, 99)), 4),
                                "pushes": len(ms)}
    res["slot_kernels"] = kernel_us()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
