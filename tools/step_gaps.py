"""Kernel times and the idle time between kernels of the C2 fused loss step, from torch.profiler's device timestamps.

    python tools/step_gaps.py [--steps 50] [--graphed]

Runs the step bench.py times -- Completionloss('cd_l2').get_loss(gen, gt) + backward on the bench's 32 x 2048 x 16384 batch
(pcn_batch, seed 0), the L2 flushed (256 MiB write) before every step -- under torch.profiler with CUDA activities, then prints
  * per kernel: launches per step and the median duration over the steps;
  * a timeline: each kernel's median first start and last end, from the end of the flush;
  * per kernel of the caller's stream, in launch order: the median interval from the end of the previous kernel on that stream
    (for the first kernel of a step, the end of the flush) to its start -- negative for a programmatic dependent dispatched early;
  * the median span of a step (flush end -> last kernel end) and how much of it no kernel on any stream covered.
--graphed profiles GraphedLossStep (the same step captured into one CUDA graph) instead of the eager call.
GENPC_LIB=<other .so> runs another build of the library (same-box A/B).  The trace goes to a temporary directory."""
import argparse
import json
import os
import re
import sys
import tempfile

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from genpc_b200.synthetic import pcn_batch  # noqa: E402
from genpc_b200.utils.loss_util import Completionloss, GraphedLossStep  # noqa: E402

B, N, M = 32, 2048, 16384


def short(name):
    name = re.sub(r"^void ", "", name)
    name = re.sub(r"\(.*$", "", name)
    name = name.replace("genpc::", "")
    if "FillFunctor" in name:
        return "torch fill"
    return name[:48]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--graphed", action="store_true")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    part, comp = pcn_batch(0, B, N, M)
    a = torch.from_numpy(part).to(dev).requires_grad_(True)
    b = torch.from_numpy(comp).to(dev).requires_grad_(True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    crit = Completionloss("cd_l2")
    if args.graphed:
        g = GraphedLossStep(crit, a.detach(), b.detach())
        step = g
    else:
        def step():
            a.grad = None
            b.grad = None
            crit.get_loss(a, b).backward()
    for _ in range(args.warmup):
        flush.zero_()
        step()
    torch.cuda.synchronize()
    acts = [torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]
    with torch.profiler.profile(activities=acts) as prof:
        for _ in range(args.steps):
            flush.zero_()
            step()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        trace = json.load(open(path))
    kern = [e for e in trace["traceEvents"] if e.get("ph") == "X" and e.get("cat") == "kernel"]
    kern.sort(key=lambda e: float(e["ts"]))
    # the flush is a fill of 256 MiB: the kernel whose duration dwarfs the rest marks the start of each step
    flush_ev = [e for e in kern if "FillFunctor" in e["name"] and float(e["dur"]) > 20.0]
    flush_ev = [e for e in flush_ev if float(e["dur"]) >= 0.5 * max(float(f["dur"]) for f in flush_ev)]
    main_stream = flush_ev[0]["args"]["stream"]
    steps = []
    for i, f in enumerate(flush_ev):
        t0 = float(f["ts"]) + float(f["dur"])
        t1 = float(flush_ev[i + 1]["ts"]) if i + 1 < len(flush_ev) else float("inf")
        steps.append((t0, [e for e in kern if t0 <= float(e["ts"]) < t1 and e is not f]))
    durs, order, gaps, spans, idle, marks = {}, None, {}, [], [], {}
    for t0, evs in steps:
        per = {}
        for e in evs:
            k = short(e["name"])
            per.setdefault(k, []).append(float(e["dur"]))
            # first start and last end of each kernel relative to the end of the flush
            m = marks.setdefault(k, {"start": [], "end": [], "stream": e["args"]["stream"] == main_stream})
            m["start"].append(float(e["ts"]) - t0)
            m["end"].append(float(e["ts"]) + float(e["dur"]) - t0)
        for k, v in per.items():
            durs.setdefault(k, []).append((len(v), sum(v)))
        mainev = [e for e in evs if e["args"]["stream"] == main_stream]
        names = tuple(short(e["name"]) for e in mainev)
        if order is None:
            order = names
        if names != order:
            continue   # a step that launched a different list (should not happen at a fixed shape)
        prev = t0
        for j, e in enumerate(mainev):
            s = float(e["ts"])
            gaps.setdefault(j, []).append(s - prev)
            prev = s + float(e["dur"])
        # idle: the part of the step no kernel (any stream) covers
        iv = sorted((float(e["ts"]), float(e["ts"]) + float(e["dur"])) for e in evs)
        end = max(b for _, b in iv)
        covered, cur_s, cur_e = 0.0, None, None
        for s, e in iv:
            if cur_e is None or s > cur_e:
                if cur_e is not None:
                    covered += cur_e - cur_s
                cur_s, cur_e = s, e
            else:
                cur_e = max(cur_e, e)
        covered += cur_e - cur_s
        spans.append(end - t0)
        idle.append(end - t0 - covered)
    print(f"C2 fused loss step ({'GraphedLossStep replay' if args.graphed else 'eager get_loss + backward'}), "
          f"{B} x {N} x {M}, {len(steps)} steps, L2 flushed before each; {torch.cuda.get_device_name(dev)}")
    print("kernel durations (us, median over steps of the per-step sum; launches per step):")
    for k, v in sorted(durs.items(), key=lambda kv: -np.median([s for _, s in kv[1]])):
        print(f"  {k:48s} {np.median([s for _, s in v]):8.2f}   x{int(np.median([n for n, _ in v]))}")
    print("timeline (us from the end of the flush, medians; a programmatic dependent starts when its first CTA is dispatched, "
          "before its predecessor ends):")
    for k, m in sorted(marks.items(), key=lambda kv: np.median(kv[1]["start"])):
        where = "" if m["stream"] else "   (another stream)"
        print(f"  {k:48s} start {np.median(m['start']):7.2f}   end {np.median(m['end']):7.2f}{where}")
    print("caller's stream, in launch order: median interval from the end of the previous kernel to the start of this one (us):")
    for j, name in enumerate(order or ()):
        print(f"  {name:48s} {np.median(gaps[j]):7.2f}")
    print(f"step span (flush end -> last kernel end): median {np.median(spans):.2f} us; "
          f"no kernel running on any stream: median {np.median(idle):.2f} us")


if __name__ == "__main__":
    main()
