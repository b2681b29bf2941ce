"""Times the mesh overlay (tepose_b200.MeshRenderer.render) on cuda:0 and prints one JSON line:

- per-frame render time at 1920x1080 for 1, 8 and 32 people, for the synthetic SMPL mesh (random vertex triples as faces: many
  frame-spanning triangles, the worst case for a rasteriser) and a closed UV sphere with SMPL's counts (6890 vertices, 13776
  faces: small triangles, as a real body mesh has).  People sit at the boxes of scripts/video_time.py, each with the camera
  crop_cam_to_frame gives a fixed crop camera.  CUDA events around each call, --warmup calls first, median (and p90) over
  --frames calls cycling through 8 frames whose boxes drift;
- next to it, a TrackedVideoTePose.push at the same number of people (slots = 32, the configuration of scripts/tracks_time.py):
  host clock around --pushes back-to-back pushes and one synchronize, per push.

The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import crop_ref, render_ref  # noqa: E402
from scripts.video_time import H, W, T, boxes, card  # noqa: E402
from tepose_b200 import MeshRenderer, TrackedVideoTePose, crop_cam_to_frame  # noqa: E402
from tepose_b200.synthetic import build_synthetic_hmr, build_synthetic_model, build_synthetic_vibe, make_smpl_model  # noqa: E402

PEOPLE = (1, 8, 32)
CROP_CAM = (0.9, 0.0, 0.1)


def meshes():
    m = make_smpl_model(0)
    sv, sf = render_ref.uv_sphere()
    return {"smpl_random_faces": (m["v_template"], m["f"]), "uv_sphere": ((0.6 * sv).astype(np.float32), sf)}


def scene(verts, P, t, dev):
    """P copies of verts at boxes(P, t), each with crop_cam_to_frame of CROP_CAM."""
    b = boxes(P, t)[:, 1:]
    cam = crop_cam_to_frame(torch.tensor([CROP_CAM] * P, dtype=torch.float64), b, W, H).float().to(dev)
    v = torch.from_numpy(np.repeat(verts[None], P, 0)).to(dev)
    return v, cam


def render_ms(r, frames, verts, P, n_frames, warmup, dev):
    scenes = [scene(verts, P, t, dev) for t in range(len(frames))]
    for i in range(warmup):
        r.render(frames[i % len(frames)], *scenes[i % len(frames)])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for i in range(n_frames):
        k = i % len(frames)
        e0.record()
        r.render(frames[k], *scenes[k])
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    drawn = float((r.render(frames[0], *scenes[0]) != frames[0]).any(-1).float().mean())
    return {"ms_median": round(float(np.median(ms)), 4), "ms_p90": round(float(np.percentile(ms, 90)), 4),
            "ms_min": round(float(min(ms)), 4), "frames": n_frames, "covered_fraction": round(drawn, 4)}


def push_ms(models, frames, P, pushes):
    tv = TrackedVideoTePose(*models, slots=32)

    def push(i):
        tv.push(frames[i % len(frames)][None], {p: tuple(row) for p, row in enumerate(boxes(P, i))})
    for i in range(T + 10):
        push(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(T + 10, T + 10 + pushes):
        push(i)
    torch.cuda.synchronize()
    return round((time.perf_counter() - t0) / pushes * 1e3, 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=200, help="timed render calls per configuration")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--pushes", type=int, default=100)
    args = ap.parse_args()
    torch.cuda.init()
    dev = "cuda:0"
    frames = [f.to(dev) for f in torch.from_numpy(crop_ref.sample_frames(1, 8, H, W))]
    res = {"card": card(), "frame": [H, W],
           "method": f"CUDA events around each render call, median over {args.frames} calls after {args.warmup} warm-up calls"}
    out = {}
    for name, (v, f) in meshes().items():
        r = MeshRenderer(f, H, W, device=dev)
        out[name] = {f"P{P}": render_ms(r, frames, v, P, args.frames, args.warmup, dev) for P in PEOPLE}
    res["render"] = out
    models = (build_synthetic_hmr(0, dev), build_synthetic_model(0, T, 1, 2048, "bf16", dev)[0],
              build_synthetic_vibe(0, T, 2, 1024, True, False, True, "bf16", dev)[0])
    res["tracked_push_ms"] = {f"P{P}": push_ms(models, frames, P, args.pushes) for P in PEOPLE}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
