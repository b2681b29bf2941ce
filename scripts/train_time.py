"""Times the training step (forward + loss + backward, no optimizer step) on cuda:0 for two configurations, in fp32 and in mixed
bf16, and prints one JSON line with the card's name and power limit read in the same run:

  released  B = 32, T = 6,  L = 2, H = 1024  (every training config the reference ships: NUM_LAYERS 2, HIDDEN_SIZE 1024)
  configs4  B = 32, T = 16, L = 1, H = 2048  (BASELINE.json configs[4])

All four (configuration, precision) models live in one process and their steps alternate, so that they see the same clocks and
neighbours.  Each step is timed alone between two CUDA events (forward + loss + backward of one batch; gradients are dropped
outside the timed region); the median over --steps steps per model is reported after --warmup untimed steps.  Inputs,
dropout masks and targets are fixed device tensors, so no host copy falls inside a step."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from tepose_b200 import synthetic as synth  # noqa: E402
from tepose_b200.train import make_dropout_masks, path_parameters  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from video_time import card  # noqa: E402

CONFIGS = {"released": dict(B=32, T=6, L=2, H=1024), "configs4": dict(B=32, T=16, L=1, H=2048)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=60, help="timed steps per configuration and precision (median reported)")
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    dev = "cuda:0"
    torch.cuda.init()
    runs = {}
    for name, c in CONFIGS.items():
        x = torch.from_numpy(synth.make_input(0, c["B"], c["T"])).to(dev)
        masks = make_dropout_masks(2 * c["B"], dev, generator=torch.Generator(device=dev).manual_seed(1234))
        tgt = {k: torch.from_numpy(v).to(dev) for k, v in synth.make_train_targets(0, 2 * c["B"]).items()}
        for precision in ("fp32", "bf16"):
            model, _ = synth.build_synthetic_model(0, c["T"], c["L"], c["H"], precision, dev)
            model.train()
            runs[(name, precision)] = (model, [p for _, p in path_parameters(model)], x, masks, tgt)

    def step(key):
        model, params, x, masks, tgt = runs[key]
        for p in params:
            p.grad = None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = model(x, is_train=True, dropout_masks=masks)[-1]
        synth.synthetic_train_loss(out, tgt).backward()
        e1.record()
        return e0, e1

    for key in runs:
        for _ in range(args.warmup):
            step(key)
    torch.cuda.synchronize()
    ms = {key: [] for key in runs}
    for _ in range(args.steps):
        for key in runs:
            e0, e1 = step(key)
            torch.cuda.synchronize()
            ms[key].append(e0.elapsed_time(e1))
    res = {"card": card(), "steps": args.steps, "warmup": args.warmup,
           "timed": "forward + loss + backward, CUDA events around each step, median over steps", "configs": CONFIGS}
    for (name, precision), t in ms.items():
        t = np.array(t)
        res[f"{name}_{precision}"] = {"ms_per_step_median": round(float(np.median(t)), 3), "ms_min": round(float(t.min()), 3),
                                      "ms_max": round(float(t.max()), 3)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
