"""Times HMR.feature_extractor at 32 crops in precision "bf16" and "fp32_tc" on cuda:0, alternating the two, and prints one
JSON line with the card's name and power limit read in the same run.

Each precision runs as one CUDA graph (GraphedHMRFeatures, what bench.py times for bf16); a round replays it --reps times between
two CUDA events, and the rounds of the two precisions alternate so that both see the same clocks and neighbours.  The weights
(~50 MB bf16, ~150 MB split) and activations exceed nothing that stays resident across a replay except the L2's 126 MB; the
crops are the same every replay.  Also printed: the features' relative L2 error against the float64 restatement
(oracle/hmr_ref.py on the same fp32 input, on the device) for both precisions."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import hmr_ref  # noqa: E402
from tepose_b200 import synthetic as psynth  # noqa: E402
from tepose_b200.graph import GraphedHMRFeatures  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from video_time import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--crops", type=int, default=32)
    ap.add_argument("--reps", type=int, default=20, help="replays per timed round")
    ap.add_argument("--rounds", type=int, default=15, help="timed rounds per precision (alternating)")
    args = ap.parse_args()
    dev = "cuda:0"
    torch.cuda.init()
    x = torch.from_numpy(psynth.make_image_batch(0, args.crops)).to(dev)
    precisions = ("bf16", "fp32_tc")
    graphs, feats = {}, {}
    for p in precisions:
        model = psynth.build_synthetic_hmr(0, dev, precision=p)
        graphs[p] = GraphedHMRFeatures(model, args.crops)
        feats[p] = graphs[p](x).clone()
    sd = {k: v.double() for k, v in model.state_dict().items() if v.is_floating_point() and not k.startswith("smpl.")}
    with torch.no_grad():
        want = hmr_ref.feature_extractor(sd, x.double())
    for p in precisions:                                    # warm-up rounds
        for _ in range(3):
            graphs[p].replay()
    torch.cuda.synchronize()
    ms = {p: [] for p in precisions}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for p in precisions:
            e0.record()
            for _ in range(args.reps):
                graphs[p].replay()
            e1.record()
            torch.cuda.synchronize()
            ms[p].append(e0.elapsed_time(e1) / args.reps)
    res = {"card": card(), "crops": args.crops, "reps_per_round": args.reps, "rounds": args.rounds}
    for p in precisions:
        t = np.array(ms[p])
        rel = float((feats[p].double() - want).norm() / want.norm())
        res[p] = {"ms_per_batch_median": round(float(np.median(t)), 4), "ms_per_batch_min": round(float(t.min()), 4),
                  "ms_per_batch_max": round(float(t.max()), 4), "us_per_crop_median": round(float(np.median(t)) * 1e3 / args.crops, 2),
                  "launches_per_replay": graphs[p].launches_per_replay, "features_rel_l2_vs_float64": rel}
    res["fp32_tc_over_bf16"] = round(res["fp32_tc"]["ms_per_batch_median"] / res["bf16"]["ms_per_batch_median"], 3)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
