"""The coarse scale sweep of reg() over a dataset of differently-sized objects: one coarse_scale_sweep_batch call (ragged ICP)
against coarse_scale_sweep called once per object (the only exact option without per-candidate point counts), and the
per-object agreement of the two.

    python tools/time_icp_ragged.py [--objects 110] [--reps 3] [--out DIR]

The objects are the seeded pairs of tools/time_registration_ragged.py: the scan (300-1400 points) is the source, the
generated shape (300-2600 points) the target, as in reg_points after voxel down-sampling; 11 scales 1.5 .. 0.8.  A host clock
around work that ends in a synchronise, after a warm-up of both forms; the two forms alternate over the repetitions.  The
card's name and power limit are read in the same run.  Writes DIR/icp_ragged.json."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from genpc_b200.reg_xyz import coarse_scale_sweep, coarse_scale_sweep_batch  # noqa: E402
from time_registration_ragged import card, dataset  # noqa: E402

SCALES = np.linspace(1.5, 0.8, 11)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--objects", type=int, default=110)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=".")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_icp_ragged: no CUDA device (this is a GPU measurement)")
    dev = torch.device("cuda:0")
    pairs = dataset(args.objects)
    sources = [torch.from_numpy(p).to(dev) for _, p in pairs]
    targets = [torch.from_numpy(c).to(dev) for c, _ in pairs]

    def batch():
        return coarse_scale_sweep_batch(sources, targets, SCALES)

    def loop():
        return [coarse_scale_sweep(s, t, SCALES, 0.075, 0.5) for s, t in zip(sources, targets)]

    batch(), loop()   # warm-up: module load, workspaces of every shape
    t_batch, t_loop = [], []
    for _ in range(args.reps):
        tb, rb = timed(batch)
        tl, rl = timed(loop)
        t_batch.append(tb)
        t_loop.append(tl)
    same_scale = [a["best_scale"] == b["best_scale"] for a, b in zip(rb, rl)]
    dloss = max(abs(a["coarse_loss"] - b["coarse_loss"]) / abs(b["coarse_loss"]) for a, b in zip(rb, rl))
    dT = max(float((a["coarse_transformation"] - b["coarse_transformation"]).abs().max()) for a, b in zip(rb, rl))
    ns = [len(p) for _, p in pairs]
    nt = [len(c) for c, _ in pairs]
    out = {
        "card": card(),
        "measured_at": time.strftime("%Y-%m-%d %H:%M:%S"),
        "objects": len(pairs), "scales": len(SCALES),
        "source_points": [min(ns), max(ns)], "target_points": [min(nt), max(nt)],
        "batch_ms": [round(t, 2) for t in t_batch],
        "per_object_loop_ms": [round(t, 2) for t in t_loop],
        "speedup_min_over_min": round(min(t_loop) / min(t_batch), 2),
        "same_best_scale": f"{sum(same_scale)}/{len(same_scale)}",
        "max_rel_loss_diff": dloss, "max_abs_transform_diff": dT,
        "agree": bool(all(same_scale) and dloss <= 1e-5 and dT <= 1e-4),
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "icp_ragged.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
