"""Times the on-device video front end (tepose_b200.VideoTePose) on cuda:0 and prints one JSON line:

- push latency at B = 1 for a 1920x1080 RGB frame: host clock around push() + synchronize, p50 / p99 over --pushes frames,
  with the frame in pinned host memory (it is uploaded inside the push) and already on the device;
- frames per second at B = 32 (32 people per frame): back-to-back pushes, one synchronize at the end;
- tp_crop_normalize_bf16 alone at N = 32 crops: CUDA events around a graph of 20 launches, and the bytes it writes.

The model is the released configuration (TePose T16 L1 H2048 bf16, VIBE L2 H1024 bootstrap) with synthetic weights; the
card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import crop_ref  # noqa: E402
from tepose_b200 import VideoTePose, _native as nv  # noqa: E402
from tepose_b200.hmr import make_crop_table  # noqa: E402
from tepose_b200.synthetic import build_synthetic_hmr, build_synthetic_model, build_synthetic_vibe  # noqa: E402

H, W, T = 1080, 1920, 16


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        out["power_limit_w"], out["max_sm_clock_mhz"] = float(q[0]), float(q[1])
    except Exception as e:                      # the numbers are still printed; the reader sees why the limit is missing
        out["power_limit_w"] = f"not read: {e}"
    return out


def boxes(B, t):
    """B people spread over the frame, drifting by a few pixels per frame."""
    rows = []
    for b in range(B):
        cx = W * (0.1 + 0.8 * ((b * 0.618) % 1.0)) + 2.5 * t
        cy = H * (0.3 + 0.4 * ((b * 0.377) % 1.0)) - 1.5 * t
        rows.append((0, cx, cy, 180 + 7 * (b % 5), 420 - 9 * (b % 4), 1.2))
    return np.array(rows)


def push_loop(vt, frames, B, n, sync_each):
    lat = []
    t0 = time.perf_counter()
    for i in range(n):
        s = time.perf_counter()
        vt.push(frames[i % len(frames)], boxes(B, i))
        if sync_each:
            torch.cuda.synchronize()
            lat.append(time.perf_counter() - s)
    torch.cuda.synchronize()
    return lat, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pushes", type=int, default=300)
    ap.add_argument("--clip", type=int, default=8, help="distinct frames cycled through")
    args = ap.parse_args()
    torch.cuda.init()
    dev = "cuda:0"
    hmr = build_synthetic_hmr(0, dev)
    model, _ = build_synthetic_model(0, T, 1, 2048, "bf16", dev)
    vibe, _ = build_synthetic_vibe(0, T, 2, 1024, True, False, True, "bf16", dev)
    host = torch.from_numpy(crop_ref.sample_frames(1, args.clip, H, W)).pin_memory()
    frames_host = [host[i:i + 1] for i in range(args.clip)]
    frames_dev = [f.to(dev) for f in frames_host]
    res = {"card": card(), "frame": [H, W], "model": "TePose T16 L1 H2048 bf16, VIBE L2 H1024 bf16, synthetic weights"}

    for where, frames in (("pinned_host", frames_host), ("device", frames_dev)):
        vt = VideoTePose(hmr, model, vibe, batch=1)
        push_loop(vt, frames, 1, T + 20, True)                         # fills the window, captures, warms up
        lat, _ = push_loop(vt, frames, 1, args.pushes, True)
        ms = np.array(lat) * 1e3
        res[f"push_B1_{where}_ms"] = {"p50": round(float(np.percentile(ms, 50)), 4), "p99": round(float(np.percentile(ms, 99)), 4),
                                      "pushes": len(ms)}
    res["launches_per_push"] = vt.launches_per_replay

    vt = VideoTePose(hmr, model, vibe, batch=32)
    push_loop(vt, frames_dev, 32, T + 20, True)
    _, secs = push_loop(vt, frames_dev, 32, args.pushes, False)
    res["B32_device_frames"] = {"frames_per_s": round(args.pushes / secs, 2), "crops_per_s": round(32 * args.pushes / secs, 1),
                                "pushes": args.pushes}

    # the crop kernel alone, N = 32, inside a graph (eager calls read the table back to check frame indices)
    N, reps = 32, 20
    table = make_crop_table(boxes(N, 0), dev)
    out = torch.empty(N, 224, 224, 4, dtype=torch.bfloat16, device=dev)
    fr = frames_dev[0]

    def launch():
        nv.check(nv.lib().tp_crop_normalize_bf16(nv.ptr(fr), 1, H, W, nv.ptr(table), N, nv.ptr(out), nv.stream()))
    launch()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            launch()
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
    us = float(np.median(times))
    written = out.numel() * out.element_size()
    res["crop_kernel_N32"] = {"us_median": round(us, 3), "us_min": round(float(min(times)), 3), "bytes_written": written,
                              "write_GBps": round(written / (us * 1e-6) / 1e9, 1),
                              "note": "the same 6.2 MB frame every launch: its taps are L2 hits after the first"}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
