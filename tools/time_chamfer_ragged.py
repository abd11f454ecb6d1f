"""Ragged Chamfer loss steps (genpc_chamfer_forward_ragged + genpc_chamfer_loss_backward_ragged): ms per
Completionloss('cd_l1') forward + backward step in three settings.

    python tools/time_chamfer_ragged.py [--reps 50] [--other-tree DIR] [--out DIR]

1. dataset: the 110 pairs of tools/time_registration_ragged.py (300-2600 x 300-1400 points), generated shape vs partial scan,
   as ONE ragged step against one step per pair (the only exact option without lengths); also checks that the ragged loss is
   the mean of the per-pair losses.
2. c2_ragged: B = 32, partial clouds of 1500-2048 points in a 2048 stride, complete clouds of 16384, against the equal-size
   step at 32 x 2048 x 16384 (which takes the pruned scan): the price of the exhaustive scan a ragged batch always runs.
3. c2_ab (with --other-tree): the unragged C2 step of this tree against another built checkout of the project (e.g. the parent
   commit), in alternating child processes of this call.

CUDA events around work that ends in a synchronise, after a warm-up; the card's name and power limit are read in the same run.
Writes DIR/chamfer_ragged.json."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
from genpc_b200.optim_registration.diff_obj_pose import pad_clouds  # noqa: E402
from genpc_b200.synthetic import pcn_batch  # noqa: E402
from genpc_b200.utils.loss_util import Completionloss  # noqa: E402
from time_registration_ragged import card, dataset  # noqa: E402


def timed(fn, reps, warmup=5):
    """ms per call of fn (CUDA events around `reps` calls, then a synchronise)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / reps


def step_fn(cl, g, t, lg=None, lt=None):
    def step():
        g.grad = None
        t.grad = None
        loss = cl.get_loss(g, t, lg, lt)
        loss.backward()
        return loss
    return step


def c2_equal(dev):
    part, comp = pcn_batch(0, 32, 2048, 16384)
    return (torch.from_numpy(part).to(dev).requires_grad_(True), torch.from_numpy(comp).to(dev).requires_grad_(True))


C2_CHILD = """
import sys, json
sys.path.insert(0, sys.argv[1])
import torch
from genpc_b200.synthetic import pcn_batch
from genpc_b200.utils.loss_util import Completionloss
dev = torch.device("cuda:0")
part, comp = pcn_batch(0, 32, 2048, 16384)
g = torch.from_numpy(part).to(dev).requires_grad_(True)
t = torch.from_numpy(comp).to(dev).requires_grad_(True)
cl = Completionloss("cd_l1")
def step():
    g.grad = None
    t.grad = None
    cl.get_loss(g, t).backward()
for _ in range(10):
    step()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
reps = int(sys.argv[2])
e0.record()
for _ in range(reps):
    step()
e1.record()
torch.cuda.synchronize()
print(json.dumps({"ms": e0.elapsed_time(e1) / reps}))
"""


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--other-tree", default=None)
    ap.add_argument("--ab-rounds", type=int, default=4)
    ap.add_argument("--out", default=".")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    res = {"card": card()}
    cl = Completionloss("cd_l1")

    # ---- 1. the 110-pair dataset: one ragged step vs one step per pair ----
    pairs = dataset(110)
    gen, gl = pad_clouds([torch.from_numpy(c).to(dev) for c, _ in pairs])   # generated shape (complete)
    gt, tl = pad_clouds([torch.from_numpy(p).to(dev) for _, p in pairs])    # partial scan
    gen.requires_grad_(True), gt.requires_grad_(True)
    solo = [(torch.from_numpy(c[None]).to(dev).requires_grad_(True), torch.from_numpy(p[None]).to(dev).requires_grad_(True))
            for c, p in pairs]
    ragged_step = step_fn(cl, gen, gt, gl, tl)
    solo_steps = [step_fn(cl, a, b) for a, b in solo]

    def per_pair():
        return [s() for s in solo_steps]

    ragged_loss = float(ragged_step().detach())
    solo_losses = [float(x.detach()) for x in per_pair()]
    mean_solo = float(np.mean(np.array(solo_losses, np.float64)))
    rs, ss = [], []
    for _ in range(3):   # alternated
        rs.append(timed(ragged_step, args.reps))
        ss.append(timed(per_pair, max(1, args.reps // 5)))
    res["dataset"] = {"pairs": len(pairs), "stride": [gen.shape[1], gt.shape[1]],
                      "ragged_ms": rs, "per_pair_ms": ss, "speedup": [s / r for s, r in zip(ss, rs)],
                      "ragged_loss": ragged_loss, "mean_of_per_pair_losses": mean_solo,
                      "rel_diff": abs(ragged_loss - mean_solo) / abs(mean_solo)}

    # ---- 2. C2-sized ragged batch vs the equal-size step ----
    g, t = c2_equal(dev)
    rng = np.random.default_rng(0)
    lg = torch.from_numpy(rng.integers(1500, 2049, size=32).astype(np.int32)).to(dev)
    eq_step, rg_step = step_fn(cl, g, t), step_fn(cl, g, t, lg, None)
    eq, rg = [], []
    for _ in range(3):
        eq.append(timed(eq_step, args.reps))
        rg.append(timed(rg_step, args.reps))
    res["c2_ragged"] = {"B": 32, "partial_stride": 2048, "partial_lengths": [int(x) for x in lg.cpu()], "complete": 16384,
                        "equal_size_ms": eq, "ragged_ms": rg}

    # ---- 3. unragged C2 step: this tree vs another checkout, alternating child processes ----
    if args.other_tree:
        ab = {"this": [], "other": []}
        for _ in range(args.ab_rounds):
            for name, root in (("this", os.path.dirname(HERE)), ("other", os.path.abspath(args.other_tree))):
                env = {k: v for k, v in os.environ.items() if k != "GENPC_LIB"}
                out = subprocess.run([sys.executable, "-c", C2_CHILD, root, str(args.reps * 4)], env=env, cwd=root,
                                     capture_output=True, text=True, check=True).stdout
                ab[name].append(json.loads(out.strip().split("\n")[-1])["ms"])
        res["c2_ab"] = ab
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "chamfer_ragged.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
