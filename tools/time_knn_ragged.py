"""The statistical outlier filter of reg_points over a dataset: one remove_statistical_outlier call on a batch of clouds
against one call per cloud (the only form before per-cloud point counts), and the per-cloud agreement of the masks.

    python tools/time_knn_ragged.py [--reps 3] [--out DIR]
    python tools/time_knn_ragged.py --ab OTHER_LIB [--rounds 3] [--out DIR]

Two seeded workloads from genpc_b200.synthetic, as reg_points calls the filter:
  (a) fused: 110 fused-size clouds of 20 000 points (FPS cuts every fused cloud to n_fused = 20 000), an equal-size batch
      called with lengths=None, std_ratio=2.5;
  (b) scans: 32 scans of 20 000-140 000 points (the pcn / kitti scans are 45 K-139 K points), a ragged batch, std_ratio=1.5.
Each cloud is a superquadric surface with 1 % of its points pushed off it, so that the filter removes some.  A host clock
around work that ends in a synchronise, after a warm-up of both forms; the two forms alternate over the repetitions.  The
card's name and power limit are read in the same run.  Writes DIR/knn_ragged.json.

--ab OTHER_LIB times the single-cloud genpc_knn_mean_distance on 20 000 and 71 372 points at k = 20 and at k = 25 and 32, the
two list sizes whose resident CTAs per SM changed with the ragged kernel (a 20 000-point cloud is under one wave at either
occupancy, a 71 372-point cloud is not), with this tree's library and with
OTHER_LIB (e.g. the parent commit's build, GENPC_LIB=OTHER_LIB), in alternating child processes; CUDA events over 20 calls,
median of 5.  Writes DIR/knn_single_ab.json."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from genpc_b200.optim_registration.diff_obj_pose import pad_clouds  # noqa: E402
from genpc_b200.reg_xyz import knn_mean_distance, remove_statistical_outlier  # noqa: E402
from genpc_b200.synthetic import superquadric  # noqa: E402
from time_registration_ragged import card  # noqa: E402

SINGLE = [(20000, 20), (71372, 20), (20000, 25), (71372, 25), (20000, 32), (71372, 32)]


def noisy_cloud(seed, n):
    x = superquadric(seed, n)
    rng = np.random.default_rng(seed + 101)
    off = rng.choice(n, n // 100, replace=False)
    x[off] += rng.normal(0, 0.05, (len(off), 3)).astype(np.float32)
    return x


def workloads():
    rng = np.random.default_rng(0)
    fused = [noisy_cloud(i, 20000) for i in range(110)]
    scans = [noisy_cloud(1000 + i, int(n)) for i, n in enumerate(rng.integers(20000, 140001, 32))]
    return {"fused": (fused, False, 2.5), "scans": (scans, True, 1.5)}


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def run_workload(dev, xs, ragged, ratio, reps):
    ts = [torch.from_numpy(x).to(dev) for x in xs]
    if ragged:
        pad, ln = pad_clouds(ts)
    else:
        pad, ln = torch.stack(ts), None

    def batch():
        return remove_statistical_outlier(pad, 20, ratio, ln)

    def loop():
        return [remove_statistical_outlier(t, 20, ratio) for t in ts]

    batch(), loop()   # warm-up: module load, both forms
    t_batch, t_loop = [], []
    for _ in range(reps):
        tb, kb = timed(batch)
        tl, kl = timed(loop)
        t_batch.append(tb)
        t_loop.append(tl)
    kb = kb.cpu()
    agree = all(torch.equal(kb[i, :len(x)], kl[i].cpu()) and not kb[i, len(x):].any() for i, x in enumerate(xs))
    ns = [len(x) for x in xs]
    return {
        "clouds": len(xs), "points": [min(ns), max(ns)], "lengths": "per cloud" if ragged else "None (equal size)",
        "std_ratio": ratio, "nb_neighbors": 20,
        "batch_ms": [round(t, 3) for t in t_batch], "per_cloud_loop_ms": [round(t, 3) for t in t_loop],
        "batch_ms_min_max": [round(min(t_batch), 3), round(max(t_batch), 3)],
        "loop_ms_min_max": [round(min(t_loop), 3), round(max(t_loop), 3)],
        "speedup_min_over_min": round(min(t_loop) / min(t_batch), 2),
        "kept_points": int(kb.sum()), "masks_agree": bool(agree),
    }


def single(dev):
    """Median ms per single-cloud genpc_knn_mean_distance call for every SINGLE case, on the library GENPC_LIB names (default:
    this tree's).  The entry is bound here on its own, so that a library built before the ragged entry existed loads too."""
    import ctypes

    from genpc_b200 import _lib

    L = ctypes.CDLL(_lib.LIB_PATH)
    fn = L.genpc_knn_mean_distance
    fn.restype, fn.argtypes = _lib._SIGNATURES["genpc_knn_mean_distance"]
    stream = _lib.current_stream(dev)
    out = {}
    for n, k in SINGLE:
        t = torch.from_numpy(noisy_cloud(7, n)).to(dev)
        md = torch.empty(n, device=dev)

        def call():
            _lib.check(fn(_lib.ptr(t), n, k, 1, _lib.ptr(md), stream), "genpc_knn_mean_distance")

        for _ in range(3):
            call()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ms = []
        for _ in range(5):
            torch.cuda.synchronize()
            e0.record()
            for _ in range(20):
                call()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1) / 20)
        out[f"n{n}_k{k}"] = round(float(np.median(ms)), 4)
    return out


def ab(other, rounds, out_dir):
    runs = {"this": [], "other": []}
    for _ in range(rounds):
        for tag in ("this", "other"):
            env = dict(os.environ)
            env.pop("GENPC_LIB", None)
            if tag == "other":
                env["GENPC_LIB"] = os.path.abspath(other)
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--single"], env=env, capture_output=True, text=True)
            if p.returncode != 0:
                raise SystemExit(f"time_knn_ragged --single ({tag}) failed:\n{p.stderr}")
            runs[tag].append(json.loads(p.stdout.strip().split("\n")[-1]))
    res = {"card": card(), "measured_at": time.strftime("%Y-%m-%d %H:%M:%S"), "other_lib": os.path.basename(other),
           "ms_per_call_median_of_5x20": runs,
           "min_max": {tag: {c: [min(r[c] for r in rs), max(r[c] for r in rs)] for c in rs[0]} for tag, rs in runs.items()}}
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "knn_single_ab.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=".")
    ap.add_argument("--ab", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--single", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_knn_ragged: no CUDA device (this is a GPU measurement)")
    dev = torch.device("cuda:0")
    if args.single:
        print(json.dumps(single(dev)))
        return
    if args.ab:
        ab(args.ab, args.rounds, args.out)
        return
    out = {"card": card(), "measured_at": time.strftime("%Y-%m-%d %H:%M:%S")}
    for name, (xs, ragged, ratio) in workloads().items():
        out[name] = run_workload(dev, xs, ragged, ratio, args.reps)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "knn_ragged.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
