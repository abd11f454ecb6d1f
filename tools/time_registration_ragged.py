"""A dataset of differently-sized cloud pairs registered in one ragged batch against one RegistrationBatch per pair (the only
exact option without per-pair point counts): ms for 4 starts x 201 Adam iterations (reg()'s iters=200 + 1), and the per-pair
agreement of the two.

    python tools/time_registration_ragged.py [--pairs 110] [--reps 3] [--out DIR]

110 seeded pairs (the size of the Waymo object set) from genpc_b200.synthetic: 300-2600 moving and 300-1400 fixed points, the
sizes after the pipeline's voxel down-sampling, none a multiple of 128.  CUDA events around work that ends in a synchronise,
after a warm-up of both forms; the card's name and power limit are read in the same run.  Writes DIR/registration_ragged.json."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from genpc_b200.optim_registration.diff_obj_pose import RegistrationBatch  # noqa: E402
from genpc_b200.synthetic import partial_view, rigid_perturb, superquadric  # noqa: E402

STARTS, ITERS = 4, 201


def dataset(n, seed=0):
    rng = np.random.default_rng(seed)
    pairs = []
    for i in range(n):
        nc, nr = 128, 128
        while nc % 128 == 0:
            nc = int(rng.integers(300, 2601))
        while nr % 128 == 0:
            nr = int(rng.integers(300, 1401))
        comp = superquadric(seed + i, nc)
        part, _ = rigid_perturb(partial_view(comp, seed + i, nr), seed + i, max_rot_deg=20.0, max_t=0.05, scale_range=(0.7, 0.9))
        pairs.append((comp, part))
    return pairs


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().split("\n")[0]
        name, power = (v.strip() for v in q.split(","))
        return {"name": name, "power_limit": power}
    except Exception as e:  # the timing stands without it, but says so
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"not read: {e}"}


def ragged(dev, pairs, iters):
    return RegistrationBatch.from_clouds([torch.from_numpy(c).to(dev) for c, _ in pairs],
                                         [torch.from_numpy(p).to(dev) for _, p in pairs], n_starts=STARTS, lr=0.01,
                                         max_iters=iters)


def solos(dev, pairs, iters):
    return [RegistrationBatch(torch.from_numpy(c[None]).to(dev), torch.from_numpy(p[None]).to(dev), n_starts=STARTS, lr=0.01,
                              max_iters=iters) for c, p in pairs]


def timed(fn):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=110)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=".")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_registration_ragged: no CUDA device (this is a GPU measurement)")
    dev = torch.device("cuda:0")
    pairs = dataset(args.pairs)
    # warm-up of both forms (module load, cooperative and per-iteration launches)
    rb = ragged(dev, pairs, 10)
    rb.run(10)
    for s in solos(dev, pairs, 10):
        s.run(10)
    torch.cuda.synchronize()
    t_ragged, t_solo = [], []
    for _ in range(args.reps):
        rb = ragged(dev, pairs, ITERS)
        t_ragged.append(timed(lambda: rb.run(ITERS)))
        ss = solos(dev, pairs, ITERS)
        t_solo.append(timed(lambda: [s.run(ITERS) for s in ss]))
    # agreement per pair: params absolute, losses relative (the partial sums are taken in another order)
    rp, rl = rb.params.cpu().numpy(), rb.losses().cpu().numpy()
    dp, dl = 0.0, 0.0
    for c, s in enumerate(ss):
        mine = slice(c * STARTS, (c + 1) * STARTS)
        sp, sl = s.params.cpu().numpy(), s.losses().cpu().numpy()
        dp = max(dp, float(np.abs(rp[mine] - sp).max()))
        dl = max(dl, float((np.abs(rl[mine] - sl) / np.abs(sl)).max()))
    nc = [len(c) for c, _ in pairs]
    nr = [len(p) for _, p in pairs]
    out = {
        "card": card(),
        "measured_at": time.strftime("%Y-%m-%d %H:%M:%S"),
        "pairs": len(pairs), "starts": STARTS, "iters": ITERS,
        "complete_points": [min(nc), max(nc)], "partial_points": [min(nr), max(nr)],
        "padded_strides": [rb.Nc, rb.Nr],
        "ragged_ms": [round(t, 3) for t in t_ragged],
        "solo_loop_ms": [round(t, 3) for t in t_solo],
        "ragged_us_per_iter": round(min(t_ragged) / ITERS * 1e3, 2),
        "solo_loop_us_per_iter": round(min(t_solo) / ITERS * 1e3, 2),
        "speedup_min_over_min": round(min(t_solo) / min(t_ragged), 2),
        "max_abs_param_diff": dp, "max_rel_loss_diff": dl,
        "agree_1e-6": bool(dp <= 1e-6 and dl <= 1e-6),
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "registration_ragged.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
