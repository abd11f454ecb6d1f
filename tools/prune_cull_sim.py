"""python tools/prune_cull_sim.py [pairs]  (CPU only, ~1 min per pair)

CPU simulation of the pruned C2 scan's block walk (nn_prune_kernel semantics) on the bench's own inputs:
how many (group, block) visits and 8-target chunks the group-box rule alone evaluates, and how many of them
the per-lane point-to-box tests (block level, chunk level; pr_visit_block in csrc/nn_prune.cuh) skip, against a
per-lane block test with a group-box chunk test.  The kernel's counters (genpc_chamfer_prune_stats: blocks walked,
chunks evaluated) are the GPU side of the same figures.  Exactness does not matter here: counts only."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from genpc_b200.synthetic import pcn_batch


def hilbert_key(x, y, z, bits):
    X = [x.copy(), y.copy(), z.copy()]
    M = 1 << (bits - 1)
    Q = M
    while Q > 1:
        P = Q - 1
        for i in range(3):
            m = (X[i] & Q) != 0
            X0 = X[0].copy()
            t = (X[0] ^ X[i]) & P
            newX0 = np.where(m, X[0] ^ P, X[0] ^ t)
            newXi = np.where(m, X[i], X[i] ^ t)
            X[0] = newX0
            if i != 0:
                X[i] = newXi
            else:
                X[0] = np.where(m, X0 ^ P, X0)  # i == 0: t == 0
        Q >>= 1
    X[1] ^= X[0]
    X[2] ^= X[1]
    t = np.zeros_like(x)
    Q = M
    while Q > 1:
        t = np.where((X[2] & Q) != 0, t ^ (Q - 1), t)
        Q >>= 1
    X = [v ^ t for v in X]
    key = np.zeros_like(x)
    for j in range(bits - 1, -1, -1):
        for i in range(3):
            key = (key << 1) | ((X[i] >> j) & 1)
    return key


def sort_cloud(p):
    n = len(p)
    bits = 4 if n >= 2048 else 3
    lo, hi = p.min(0), p.max(0)
    sc = (1 << bits) / np.maximum(hi - lo, 1e-30)
    cc = np.clip(((p - lo) * sc).astype(np.int64), 0, (1 << bits) - 1)
    key = hilbert_key(cc[:, 0], cc[:, 1], cc[:, 2], bits)
    return p[np.argsort(key, kind="stable")]


def boxes(p, size):
    k = len(p) // size
    q = p[: k * size].reshape(k, size, 3)
    return q.min(1), q.max(1)


def box_d2(lo1, hi1, lo2, hi2):
    d = np.maximum(np.maximum(lo2 - hi1, lo1 - hi2), 0)
    return (d * d).sum(-1)


def walk(Q, T):
    """Q, T sorted; returns counters."""
    blo, bhi = boxes(T, 64)
    clo, chi = boxes(T, 8)
    nblk = len(blo)
    c = dict(groups=0, visits=0, visits_needed=0, chunks_needed=0, chunks_groupbox=0)
    for g in range(len(Q) // 32):
        q = Q[g * 32:(g + 1) * 32]
        glo, ghi = q.min(0), q.max(0)
        bd = box_d2(glo[None], ghi[None], blo, bhi) * 0.99999
        order = np.argsort(bd, kind="stable")
        best = np.full(32, np.inf)
        c["groups"] += 1
        for blk in order:
            if not bd[blk] <= best.max():
                break
            c["visits"] += 1
            # per-lane point-to-block-box distance against the lane's own running minimum
            pl = box_d2(q, q, blo[blk][None], bhi[blk][None]) * 0.99999
            if np.any(pl <= best):
                c["visits_needed"] += 1
                thr = best.max()
                gd = box_d2(glo[None], ghi[None], clo[blk * 8:blk * 8 + 8], chi[blk * 8:blk * 8 + 8]) * 0.99999
                c["chunks_groupbox"] += int((gd <= thr).sum())
                for ch in range(blk * 8, blk * 8 + 8):
                    pc = box_d2(q, q, clo[ch][None], chi[ch][None]) * 0.99999
                    if np.any(pc <= best):
                        c["chunks_needed"] += 1
                        t = T[ch * 8:(ch + 1) * 8]
                        d = ((q[:, None, :] - t[None]) ** 2).sum(-1).min(1)
                        best = np.minimum(best, d)
            # (a skipped block / chunk cannot lower any lane's minimum: best is the same as in the current walk)
    c["blocks"] = nblk
    return c


def main():
    nb = int(sys.argv[1]) if len(sys.argv) > 1 else 4
    part, comp = pcn_batch(0, nb, 2048, 16384)
    tot = {}
    for b in range(nb):
        P, C = sort_cloud(part[b].astype(np.float64)), sort_cloud(comp[b].astype(np.float64))
        for name, (Q, T) in (("A complete->partial", (C, P)), ("B partial->complete", (P, C))):
            c = walk(Q, T)
            t = tot.setdefault(name, dict.fromkeys(c, 0))
            for k, v in c.items():
                t[k] += v
    for name, t in tot.items():
        g = t["groups"]
        print(f"{name}: {t['blocks'] // nb} blocks/cloud, visits/group {t['visits'] / g:.2f}, "
              f"block-needed/group {t['visits_needed'] / g:.2f}, chunks evaluated/group now {8 * t['visits'] / g:.1f} "
              f"-> with per-lane block+chunk culling {t['chunks_needed'] / g:.1f} ({t['chunks_needed'] / (8 * t['visits']):.1%}); "
              f"per-lane block + group-box chunk test {t['chunks_groupbox'] / g:.1f} ({t['chunks_groupbox'] / (8 * t['visits']):.1%})")


if __name__ == "__main__":
    main()
