"""icp_step_kernel (genpc_icp_step, genpc_icp_step_ragged) against a float64 Kabsch reference (oracle.icp) where Horn's
quaternion form and Kabsch/SVD can part: rotations near and at pi (quaternion w -> 0), planar, collinear and symmetric inlier
sets, exactly three inliers, a mirrored copy, clouds far from the origin, non-rigid start transforms; and at the edges of the
inlier and convergence tests.  The step-level cases call the C entries with hand-built cur / dist / idx, so they do not depend
on the Chamfer kernels, and the reference steps from the kernel's previous T.

Unique optimum (decided here in float64: the gap between the top two eigenvalues of Horn's N(H) is at least 1e-6 of the top
one): every entry of T within 2 fp32 ulps of (M_kabsch @ T_prev) rounded to float32.  The ulp is taken at the entry's
magnitude, floored at 1e-6 of the sum of the magnitudes of the terms that make the entry, so that an entry which cancels to
about 0 is held to the precision its terms allow.  While the kernel accumulated raw moments about the origin, H = sum s q^T
- cnt ms mq^T cancelled far from it: on a B200 the step was 126 ulps off at an offset of 1000 and an extent of 0.01, 2 at
an extent of 0.1 and 1 at offset 100, extent 0.01.  It now accumulates about the candidate's target row 0, and every
unique-optimum case of this file comes within 0.002 ulp there.  Not unique (collinear, symmetric, one- and two-point targets): [R|t] = T_new T_prev^-1 is a proper
rotation and reaches the Kabsch cost.  Statistics and convergence follow oracle.icp.icp_step's rules (fitness / rmse to
rtol 2e-7)."""
import ctypes
import math

import numpy as np
import pytest

import oracle
from oracle import icp as OI
from test_oracle_icp import rot
from util import shape_cloud

F32 = np.float32
BIG = 1e30            # a max_dist2 every finite dist is below
BASE = (np.random.default_rng(7).standard_normal((160, 3)) * np.array([1.0, 0.6, 0.3])).astype(F32)  # distinct axes


# ---- float64 reference -------------------------------------------------------------------------------------------------

def horn_n(s, q):
    """Horn's symmetric 4x4 N(H) of the centred cross-covariance H = sum (s - ms)(q - mq)^T (float64)."""
    s, q = np.asarray(s, np.float64), np.asarray(q, np.float64)
    H = (s - s.mean(0)).T @ (q - q.mean(0))
    (a, b, c), (d, e, f), (g, h, i) = H
    return np.array([[a + e + i, f - h, g - c, b - d],
                     [f - h, a - e - i, b + d, g + c],
                     [g - c, b + d, -a + e - i, f + h],
                     [b - d, g + c, f + h, -a - e + i]])


def relative_gap(s, q):
    ev = np.linalg.eigvalsh(horn_n(s, q))
    return (ev[-1] - ev[-2]) / abs(ev[-1]) if ev[-1] != 0 else 0.0   # N(H) = 0: every rotation is optimal


def inliers(dist, idx, nt, max_dist2):
    return (np.asarray(dist, F32) < F32(max_dist2)) & (idx >= 0) & (idx < nt)


def ulps_from_kabsch(T, s, q, T_prev):
    """max over the 12 entries of |T - round32(M_kabsch @ T_prev)| in fp32 ulps of the entry (see the module docstring)."""
    s64, q64, Tp = np.asarray(s, np.float64), np.asarray(q, np.float64), np.asarray(T_prev, np.float64)
    R, t = OI.kabsch(s64, q64)
    M = np.eye(4)
    M[:3, :3], M[:3, 3] = R, t
    ref32 = (M @ Tp)[:3].astype(F32)
    A = np.abs(M)
    A[:3, 3] = np.abs(q64.mean(0)) + np.abs(R) @ np.abs(s64.mean(0))   # the terms of t = mq - R ms
    floor = (1e-6 * (A @ np.abs(Tp))[:3]).astype(F32)
    ulp = np.spacing(np.maximum(np.abs(ref32), floor)).astype(np.float64)
    return float((np.abs(np.asarray(T, np.float64)[:3] - ref32) / ulp).max())


def nearest_rotation(A):
    U, _, Vt = np.linalg.svd(A)
    return U @ np.diag([1.0, 1.0, np.linalg.det(U @ Vt)]) @ Vt


def check_not_unique(T, s, q, T_prev):
    """[R|t] = T T_prev^-1: a proper rotation whose cost sum |R s + t - q|^2 is the Kabsch cost.  The cost is taken at the
    rotation nearest to R: R's fp32 rounding (checked by the orthogonality bound) would move it to first order where the fit
    is not exact, e.g. a one-point target."""
    s64, q64 = np.asarray(s, np.float64), np.asarray(q, np.float64)
    Rt = np.asarray(T, np.float64) @ np.linalg.inv(np.asarray(T_prev, np.float64))
    R, t = Rt[:3, :3], Rt[:3, 3]
    assert abs(np.linalg.det(R) - 1.0) <= 1e-6 and np.linalg.norm(R @ R.T - np.eye(3)) <= 1e-6, R
    Rk, tk = OI.kabsch(s64, q64)
    cost = ((s64 @ nearest_rotation(R).T + t - q64) ** 2).sum()
    best = ((s64 @ Rk.T + tk - q64) ** 2).sum()
    assert cost <= best + 1e-9 * ((s64 - s64.mean(0)) ** 2).sum(), (cost, best)


# ---- C entries ---------------------------------------------------------------------------------------------------------

def dev_tensors(dev, *arrays):
    import torch

    return [None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in arrays]


def icp_step(dev, cur, target, dist, idx, T, state, max_dist2, rel_f=1e-6, rel_r=1e-6, update=1):
    """genpc_icp_step on numpy inputs: cur [K,Ns,3], target [Kt,Nt,3], dist / idx [K,Ns], T [K,4,4], state [K,4]
    -> (T, state) as numpy."""
    import torch

    from genpc_b200 import _lib

    c, tg, d, i, Tt, st = dev_tensors(dev, cur, target, dist, idx, T, state)
    K, Ns, Kt, Nt = cur.shape[0], cur.shape[1], target.shape[0], target.shape[1]
    rc = _lib.lib().genpc_icp_step(_lib.ptr(c), _lib.ptr(tg), _lib.ptr(d), _lib.ptr(i), _lib.ptr(Tt), _lib.ptr(st), K, Ns, Kt,
                                   Nt, float(max_dist2), float(rel_f), float(rel_r), int(update), _lib.current_stream(dev))
    assert rc == 0
    torch.cuda.synchronize()
    return Tt.cpu().numpy(), st.cpu().numpy()


def icp_step_ragged(dev, source, cur, target, dist, idx, src_len, tgt_len, T, state, max_dist2, rel_f=1e-6, rel_r=1e-6,
                    update=1):
    """genpc_icp_step_ragged on numpy inputs (dist = idx = None: transform only) -> (T, state, cur, scan_len) as numpy."""
    import torch

    from genpc_b200 import _lib

    s, c, tg, d, i, sl, tl, Tt, st = dev_tensors(dev, source, cur, target, dist, idx, np.asarray(src_len, np.int32),
                                                 np.asarray(tgt_len, np.int32), T, state)
    scan_len = torch.full((source.shape[0],), -99, dtype=torch.int32, device=dev)
    K, Ns, Kt, Nt = source.shape[0], source.shape[1], target.shape[0], target.shape[1]
    rc = _lib.lib().genpc_icp_step_ragged(_lib.ptr(s), _lib.ptr(c), _lib.ptr(tg), _lib.ptr(d), _lib.ptr(i), _lib.ptr(sl),
                                          _lib.ptr(tl), _lib.ptr(scan_len), _lib.ptr(Tt), _lib.ptr(st), K, Ns, Kt, Nt,
                                          float(max_dist2), float(rel_f), float(rel_r), int(update), _lib.current_stream(dev))
    assert rc == 0
    torch.cuda.synchronize()
    return Tt.cpu().numpy(), st.cpu().numpy(), c.cpu().numpy(), scan_len.cpu().numpy()


def bits(a):
    return np.ascontiguousarray(a, F32).view(np.int32)


def transform_rows(T, source):
    """cur = T source in the kernel's documented order: c_r = fma(T[r][2], z, fma(T[r][1], y, fma(T[r][0], x, T[r][3])))."""
    x, y, z = source[:, 0], source[:, 1], source[:, 2]
    return np.stack([oracle.fmaf(T[r, 2], z, oracle.fmaf(T[r, 1], y, oracle.fmaf(T[r, 0], x, T[r, 3]))) for r in range(3)], 1)


# ---- cases -------------------------------------------------------------------------------------------------------------

def rigid(R, t=(0.0, 0.0, 0.0), S=(1.0, 1.0, 1.0)):
    T = np.eye(4)
    T[:3, :3], T[:3, 3] = np.asarray(R) @ np.diag(S), t
    return T.astype(F32)


def case(q, R=np.eye(3), centre=(0.0, 0.0, 0.0), noise=1e-4, T_prev=np.eye(4), seed=1, shuffle=True):
    """One candidate: target q (float32), cur = R^T (q - centre) + centre + noise, so that the optimum rotates about centre by
    ~R; the target rows are shuffled and idx follows them.  -> dict(cur, target, dist, idx, T)."""
    rng = np.random.default_rng(seed)
    q = np.asarray(q, F32)
    c = np.asarray(centre, np.float64)
    ext = max(float(np.abs(q - c).max()), 1e-30)
    s = ((q - c) @ np.asarray(R) + c + noise * ext * rng.standard_normal(q.shape)).astype(F32)
    perm = rng.permutation(len(q)) if shuffle else np.arange(len(q))
    target = q[perm]
    idx = np.argsort(perm).astype(np.int32)       # target[idx[j]] == q[j]
    dist = ((s.astype(np.float64) - q) ** 2).sum(1).astype(F32)
    return dict(cur=s, target=target, dist=dist, idx=idx, T=np.asarray(T_prev, F32))


def at(centre, extent):
    return (np.asarray(centre, np.float64) + extent * BASE.astype(np.float64)).astype(F32)


Z, OBL = [0, 0, 1], [1, 2, 3]


def unique_cases():
    out = {}
    for axis_name, axis in (("z", Z), ("oblique", OBL)):
        for ang_name, ang in (("0", 0.0), ("1e-7", 1e-7), ("pi/2", math.pi / 2), ("pi-1e-6", math.pi - 1e-6), ("pi", math.pi)):
            out[f"rotation {ang_name} about {axis_name}"] = case(BASE, rot(axis, ang) if ang else np.eye(3), noise=1e-4)
    planar = BASE * F32([1, 1, 0])
    out["planar"] = case(planar, rot(OBL, 0.7), noise=0.0)
    three = case(BASE, rot(OBL, 0.4))
    three["dist"][3:] = F32(4.0)                                  # rows 3.. are no inliers at max_dist2 = 1
    out["exactly three inliers"] = dict(three, max_dist2=1.0)
    n = np.array([1.0, -0.5, 0.8]) / np.linalg.norm([1.0, -0.5, 0.8])
    mirror = case(BASE, np.eye(3) - 2 * np.outer(n, n), noise=0.0)
    out["mirrored copy"] = mirror
    for off in (10, 100, 1000):
        for ext in (1.0, 0.1, 0.01):
            centre = np.array([1.0, -0.5, 0.3]) * off
            out[f"offset {off} extent {ext}"] = case(at(centre, ext), rot(OBL, 0.3), centre=centre)
    Rp, tp = rot([2, -1, 0.5], 0.6), (0.3, -0.2, 0.1)
    for name, S in (("diag(0.8)", (0.8,) * 3), ("diag(1.5)", (1.5,) * 3), ("diag(1.1, 1.0, 0.9)", (1.1, 1.0, 0.9))):
        out[f"start T = rotation . {name}"] = case(BASE, rot(OBL, 0.4), T_prev=rigid(Rp, tp, S))
    far = case(at(np.array([100.0, 50.0, -80.0]), 1.0), rot(OBL, 0.3), centre=(100.0, 50.0, -80.0))
    far["target"] = np.concatenate([np.full((1, 3), np.nan, F32), far["target"]])
    far["idx"] = far["idx"] + 1
    out["target row 0 NaN, never a correspondence"] = far
    return out


def not_unique_cases():
    rng = np.random.default_rng(11)
    d = np.array([0.3, -0.8, 0.5]) / np.linalg.norm([0.3, -0.8, 0.5])
    line = (rng.uniform(-1, 1, (40, 1)) * d + np.array([0.2, 0.1, -0.3])).astype(F32)
    octa = np.concatenate([np.eye(3), -np.eye(3)]).astype(F32)
    oc = dict(cur=octa, target=octa, idx=np.array([3, 1, 2, 0, 4, 5], np.int32), dist=np.full(6, 0.5, F32),
              T=np.eye(4, dtype=F32))                              # +x <-> -x: H = diag(-2, 2, 2), N(H) has a triple top
    src = BASE[:30]
    one = dict(cur=src, target=np.array([[0.3, -0.1, 0.2]], F32), idx=np.zeros(30, np.int32), dist=np.full(30, 0.5, F32),
               T=rigid(rot(OBL, 0.2), (0.1, 0, 0), (1.5, 1.5, 1.5)))
    two = dict(one, target=np.array([[0.3, -0.1, 0.2], [-0.4, 0.5, 0.1]], F32), idx=(np.arange(30) % 2).astype(np.int32))
    return {"collinear": case(line, rot(OBL, 0.9), noise=0.0), "octahedron onto a reflection of itself": oc,
            "one-point target": one, "two-point target": two}


def run_case(dev, c, rel_f=1e-6, rel_r=1e-6, update=1, state=None):
    """Both C entries on one candidate -> (T, state, oracle T) from the equal-size entry, its statistics checked against
    oracle.icp.icp_step.  The ragged entry gives bit for bit the same, except that a candidate entering converged keeps its
    fitness and rmse there."""
    state = np.zeros(4, F32) if state is None else np.asarray(state, F32)
    md2 = c.get("max_dist2", BIG)
    T, st = icp_step(dev, c["cur"][None], c["target"][None], c["dist"][None], c["idx"][None], c["T"][None], state[None], md2,
                     rel_f, rel_r, update)
    ns, nt = len(c["cur"]), len(c["target"])
    Tr, str_, _, scan = icp_step_ragged(dev, c["cur"][None], c["cur"][None], c["target"][None], c["dist"][None], c["idx"][None],
                                        [ns], [nt], c["T"][None], state[None], md2, rel_f, rel_r, update)
    assert np.array_equal(bits(T), bits(Tr))
    frozen = np.array([state[0], state[1], 1, state[3] + 1], F32) if state[2] else st[0]
    assert np.array_equal(bits(str_[0]), bits(frozen)), (str_, frozen)
    assert scan[0] == (0 if st[0, 2] else ns)
    To, so = OI.icp_step(c["cur"], c["target"], c["dist"], c["idx"], c["T"], state, md2, rel_f, rel_r, bool(update))
    assert np.allclose(st[0, :2], so[:2], rtol=2e-7, atol=1e-9), (st[0], so)
    assert st[0, 2] == so[2] and st[0, 3] == so[3], (st[0], so)
    assert np.array_equal(T[0, 3], c["T"][3])                     # the last row is never written
    return T[0], st[0], To


# ---- CPU ---------------------------------------------------------------------------------------------------------------

def test_oracle_fmaf_rounds_once():
    """oracle.fmaf is a * b + c rounded once to fp32: within half an ulp of the exact value, and unlike the two-rounding form
    where a * b loses its low bits."""
    from fractions import Fraction

    rng = np.random.default_rng(3)
    a, b, c = (rng.standard_normal(500).astype(F32) * F32(10.0) ** rng.integers(-3, 4, 500).astype(F32) for _ in range(3))
    r = oracle.fmaf(a, b, c)
    for ai, bi, ci, ri in zip(a, b, c, r):
        err = abs(Fraction(float(ai)) * Fraction(float(bi)) + Fraction(float(ci)) - Fraction(float(ri)))
        assert err <= Fraction(float(np.spacing(abs(ri)))) / 2, (ai, bi, ci, ri)
    x = F32(1 + 2.0 ** -12)            # x * x = 1 + 2^-11 + 2^-24: the 2^-24 is lost when the product is rounded first
    assert oracle.fmaf(x, x, F32(-(1 + 2.0 ** -11))) == F32(2.0 ** -24)
    assert F32(x * x) + F32(-(1 + 2.0 ** -11)) == 0
    assert oracle.fmaf([1.0, 2.0], 3.0, 0.5).tolist() == [3.5, 6.5]


def test_equal_size_entry_arguments_without_a_device():
    """K = 0 is a no-op that returns GENPC_OK before any CUDA call; K < 0, Kt not in {1, K} and sizes <= 0 are
    GENPC_ERR_SHAPE."""
    from genpc_b200 import _lib

    L = _lib.lib()
    buf = (ctypes.c_int * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)   # never dereferenced

    def step(K=2, Ns=8, Kt=2, Nt=8):
        return L.genpc_icp_step(p, p, p, p, p, p, K, Ns, Kt, Nt, 0.01, 1e-6, 1e-6, 1, None)

    assert step(K=0, Kt=1) == 0 and step(K=0, Kt=0) == 0
    assert list(buf) == [0] * 64
    assert step(K=-1, Kt=1) == -1 and step(Kt=3) == -1 and step(K=3, Kt=2) == -1
    for bad in (dict(Ns=0), dict(Ns=-3), dict(Nt=0), dict(Nt=-1)):
        assert step(**bad) == -1, bad


def test_reference_cases_are_what_they_claim():
    """The unique-optimum cases have a top-eigenvalue gap of N(H) of at least 1e-6, the others of (about) 0."""
    for name, c in unique_cases().items():
        inl = inliers(c["dist"], c["idx"], len(c["target"]), c.get("max_dist2", BIG))
        assert relative_gap(c["cur"][inl], c["target"][c["idx"][inl]]) >= 1e-6, name
    for name, c in not_unique_cases().items():
        assert relative_gap(c["cur"], c["target"][c["idx"]]) < 1e-9, name


# ---- GPU: one step -----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", list(unique_cases()))
def test_unique_optimum_within_two_ulps_of_kabsch(cuda, name):
    c = unique_cases()[name]
    T, st, To = run_case(cuda, c)
    inl = inliers(c["dist"], c["idx"], len(c["target"]), c.get("max_dist2", BIG))
    assert st[2] == 0 and st[3] == 1
    assert ulps_from_kabsch(T, c["cur"][inl], c["target"][c["idx"][inl]], c["T"]) <= 2.0, (name, T, To)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(not_unique_cases()))
def test_not_unique_optimum_reaches_the_kabsch_cost(cuda, name):
    c = not_unique_cases()[name]
    T, _, _ = run_case(cuda, c)
    check_not_unique(T, c["cur"], c["target"][c["idx"]], c["T"])


@pytest.mark.gpu
def test_inlier_edges(cuda):
    """dist == max_dist2 exactly (the rule is strict), NaN and +inf dist, idx = -1 and idx >= Nt are no inliers; the step is
    the Kabsch step of the rest.  Exactly two inliers leave T alone, exactly three update it."""
    c = case(BASE[:40], rot(OBL, 0.5))
    md2 = F32(0.3)                                  # the float32 value the kernel compares with
    c["dist"] = np.full(40, np.nextafter(md2, F32(0)), F32)
    c["dist"][0:4] = md2
    c["dist"][4:6] = np.nan
    c["dist"][6] = np.inf
    c["dist"][7] = np.nextafter(md2, F32(np.inf))
    c["idx"][8], c["idx"][9], c["idx"][10] = -1, 40, np.iinfo(np.int32).max
    c["max_dist2"] = float(md2)
    T, st, _ = run_case(cuda, c)
    keep = np.arange(11, 40)
    assert st[0] == F32(29 / 40)
    assert ulps_from_kabsch(T, c["cur"][keep], c["target"][c["idx"][keep]], c["T"]) <= 2.0
    for n_in, moves in ((2, False), (3, True)):
        d = dict(c, dist=np.where(np.arange(40) < 11 + n_in, c["dist"], F32(1.0)).astype(F32))
        T, st, _ = run_case(cuda, d)
        assert st[0] == F32(n_in / 40) and np.array_equal(T, c["T"]) != moves, n_in


@pytest.mark.gpu
def test_convergence_edges(cuda):
    """|delta fitness| or |delta rmse| equal to its threshold is not convergence (strict <), one fp32 step closer on both is;
    the first call never converges; a converged candidate and update = 0 leave T alone while the statistics move."""
    c = case(BASE, rot(OBL, 0.2))
    c["dist"] = np.where(np.arange(160) < 80, F32(0.25), F32(4.0)).astype(F32)   # fitness 0.5, rmse 0.5 exactly
    c["max_dist2"] = 1.0
    thr = 2.0 ** -10
    lo, hi = F32(0.5 - thr), F32(0.5 + thr)                         # |0.5 - lo| == |0.5 - hi| == thr exactly
    lo_in, hi_in = np.nextafter(lo, F32(1)), np.nextafter(hi, F32(0))
    for st0, converges in (([lo, 0.5, 0, 1], False), ([0.5, hi, 0, 1], False), ([lo, hi, 0, 1], False),
                           ([hi, lo, 0, 1], False), ([lo_in, hi_in, 0, 1], True), ([hi_in, lo_in, 0, 1], True),
                           ([0.5, 0.5, 0, 0], False), ([0.1, 0.9, 1, 7], True)):
        T, st, _ = run_case(cuda, c, rel_f=thr, rel_r=thr, state=st0)
        assert (st[0], st[1], st[2], st[3]) == (0.5, 0.5, float(converges), st0[3] + 1), (st0, st)
        assert np.array_equal(T, c["T"]) == converges, st0
    T, st, _ = run_case(cuda, c, update=0)
    assert np.array_equal(T, c["T"]) and st[0] == 0.5 and st[3] == 1


# ---- GPU: a shared target, bit for bit ---------------------------------------------------------------------------------

def shared_target_batch(K=5, Ns=96, Nt=120, seed=4):
    rng = np.random.default_rng(seed)
    tgt = shape_cloud(seed, 1, Nt)[0]
    cur = np.stack([(tgt[rng.permutation(Nt)[:Ns]] @ rot(rng.standard_normal(3), 0.3 * k)).astype(F32) for k in range(K)])
    idx = rng.integers(0, Nt, (K, Ns)).astype(np.int32)
    dist = rng.uniform(0, 0.02, (K, Ns)).astype(F32)
    T = np.stack([rigid(rot(rng.standard_normal(3), 0.2), rng.standard_normal(3) * 0.1, (1.0 + 0.1 * k,) * 3) for k in range(K)])
    return tgt, cur, dist, idx, T


@pytest.mark.gpu
def test_shared_target_equals_the_replicated_target(cuda):
    """Kt = 1 reads target row block 0 for every candidate: T and state bit for bit those of the same call on K copies.  The
    shared target sits at the start of a K-block buffer whose other blocks are NaN."""
    tgt, cur, dist, idx, T = shared_target_batch()
    K, Nt = cur.shape[0], tgt.shape[0]
    state = np.zeros((K, 4), F32)
    rep = icp_step(cuda, cur, np.repeat(tgt[None], K, 0), dist, idx, T, state, 0.01)
    buf = np.full((K, Nt, 3), np.nan, F32)
    buf[0] = tgt
    import torch

    from genpc_b200 import _lib

    c, b, d, i, Tt, st = dev_tensors(cuda, cur, buf, dist, idx, T, state)
    assert _lib.lib().genpc_icp_step(_lib.ptr(c), _lib.ptr(b), _lib.ptr(d), _lib.ptr(i), _lib.ptr(Tt), _lib.ptr(st), K,
                                     cur.shape[1], 1, Nt, 0.01, 1e-6, 1e-6, 1, _lib.current_stream(cuda)) == 0
    torch.cuda.synchronize()
    assert np.array_equal(bits(Tt.cpu().numpy()), bits(rep[0])) and np.array_equal(bits(st.cpu().numpy()), bits(rep[1]))
    assert not np.array_equal(rep[0], T)          # the step did move the candidates


@pytest.mark.gpu
def test_ragged_shared_target_equals_the_replicated_target(cuda):
    """Ragged entry, Kt = 1: tgt_len[0] is every candidate's target length (tgt_len[1:] hold other values), per-candidate
    source lengths 0 .. Ns, NaN padding: T, state, cur and scan_len bit for bit those of K copies of the target, for the
    transform-only call and a step whose idx also points past tgt_len[0]."""
    import torch

    from genpc_b200 import _lib

    tgt, cur, dist, idx, T = shared_target_batch()
    K, Ns = cur.shape[:2]
    Nt, nt0 = tgt.shape[0], 100
    src_len = np.array([Ns, 37, 0, 3, 95], np.int32)
    idx[:, ::7] = nt0 + 5                          # past tgt_len[0], inside the stride: no inlier
    source = cur.copy()
    for k, n in enumerate(src_len):
        source[k, n:] = cur[k, n:] = np.nan
        dist[k, n:] = np.nan
        idx[k, n:] = -123
    rep_t = np.full((K, Nt, 3), np.nan, F32)
    rep_t[:, :nt0] = tgt[:nt0]
    one_t = np.full((K, Nt, 3), np.nan, F32)       # a K-block buffer: a wrong block offset reads NaN, not unowned memory
    one_t[0, :nt0] = tgt[:nt0]
    lens_rep = np.full(K, nt0, np.int32)
    lens_one = np.array([nt0, Nt, 0, -7, 10 ** 6], np.int32)

    def run(target, lens, Kt, d, i, cur_in, T_in, st_in):
        s, c, tg, dd, ii, sl, tl, Tt, st = dev_tensors(cuda, source, cur_in, target, d, i, src_len, lens, T_in, st_in)
        scan = torch.full((K,), -99, dtype=torch.int32, device=cuda)
        assert _lib.lib().genpc_icp_step_ragged(_lib.ptr(s), _lib.ptr(c), _lib.ptr(tg), _lib.ptr(dd), _lib.ptr(ii),
                                                _lib.ptr(sl), _lib.ptr(tl), _lib.ptr(scan), _lib.ptr(Tt), _lib.ptr(st), K, Ns,
                                                Kt, Nt, 0.01, 1e-6, 1e-6, 1, _lib.current_stream(cuda)) == 0
        torch.cuda.synchronize()
        return Tt.cpu().numpy(), st.cpu().numpy(), c.cpu().numpy(), scan.cpu().numpy()

    state = np.zeros((K, 4), F32)
    sentinel = np.full_like(cur, 7.5e33)
    for d, i, cur_in in ((None, None, sentinel), (dist, idx, cur)):
        a = run(rep_t, lens_rep, K, d, i, cur_in, T, state)
        b = run(one_t, lens_one, 1, d, i, cur_in, T, state)
        for x, y in zip(a, b):
            assert np.array_equal(np.ascontiguousarray(x).view(np.int32), np.ascontiguousarray(y).view(np.int32))
    assert not np.array_equal(a[0][0], T[0]) and not np.array_equal(a[0][4], T[4])   # the step did move them


# ---- GPU: the ragged cur write, bit for bit ----------------------------------------------------------------------------

@pytest.mark.gpu
def test_ragged_cur_write_follows_the_documented_fma_order(cuda):
    """cur[k, j] = T_k source[k, j] for j < src_len[k], c_r = fma(T[r][2], z, fma(T[r][1], y, fma(T[r][0], x, T[r][3]))),
    bit for bit: after a transform-only call (T untouched, scan_len = 0 for a converged candidate) and after a step (with the
    new T).  Rows past src_len, candidates with 0 source or 0 target points and a candidate that enters converged are left
    as they were."""
    rng = np.random.default_rng(8)
    K, Ns, Nt = 6, 300, 200
    tgt = (rng.standard_normal((K, Nt, 3)) * 0.4).astype(F32)
    source = (rng.standard_normal((K, Ns, 3)) * np.float32(3.0)).astype(F32)
    T = np.stack([rigid(rot(rng.standard_normal(3), 1.3 * k), rng.standard_normal(3) * 5, (0.8, 1.5, 1.1)) for k in range(K)])
    src_len = np.array([Ns, 211, 0, 1, 77, 150], np.int32)
    tgt_len = np.array([Nt, 120, 50, 9, 0, 60], np.int32)
    state = np.zeros((K, 4), F32)
    state[5] = [0.9, 0.01, 1, 3]                                 # enters converged
    sentinel = F32(-7.25e31)
    cur0 = np.full((K, Ns, 3), sentinel, F32)
    written = [k for k in range(K) if src_len[k] > 0 and tgt_len[k] > 0]

    def expect(Tn, before, skip=()):
        want = before.copy()
        for k in written:
            if k not in skip:
                want[k, :src_len[k]] = transform_rows(Tn[k], source[k, :src_len[k]])
        return want

    T1, st1, cur1, scan1 = icp_step_ragged(cuda, source, cur0, tgt, None, None, src_len, tgt_len, T, state, 0.01)
    assert np.array_equal(bits(T1), bits(T)) and np.array_equal(bits(st1), bits(state))
    assert scan1.tolist() == [int(n) if k != 5 else 0 for k, n in enumerate(src_len)]
    assert np.array_equal(bits(cur1), bits(expect(T, cur0)))
    # a step from cur = T source with nearest neighbours by brute force: every moving candidate gets its new T's rows
    dist = np.full((K, Ns), np.nan, F32)
    idx = np.full((K, Ns), -1, np.int32)
    for k in written:
        n, m = src_len[k], tgt_len[k]
        d2 = ((cur1[k, :n, None].astype(np.float64) - tgt[k, None, :m]) ** 2).sum(-1)
        idx[k, :n] = d2.argmin(1)
        dist[k, :n] = d2.min(1)
    T2, st2, cur2, scan2 = icp_step_ragged(cuda, source, cur1, tgt, dist, idx, src_len, tgt_len, T1, st1, 1e6)
    assert np.array_equal(bits(T2[5]), bits(T[5])) and not np.array_equal(T2[0], T[0])
    assert np.array_equal(bits(cur2), bits(expect(T2, cur1, skip=(5,))))


# ---- GPU: whole loops --------------------------------------------------------------------------------------------------

def clusters(seed, n):
    """Six separated blobs of different sizes: no symmetry, and an ICP from a large rotation settles in a few iterations."""
    rng = np.random.default_rng(seed)
    cen = rng.standard_normal((6, 3)) * 0.3
    size = np.array([0.02, 0.03, 0.05, 0.04, 0.06, 0.025])
    lab = rng.integers(0, 6, n)
    return (cen[lab] + rng.standard_normal((n, 3)) * size[lab, None]).astype(F32)


@pytest.mark.gpu
def test_large_rotation_loops_vs_the_oracle(cuda):
    """A 2.75 rad rotation of a non-symmetric cloud, max_correspondence_distance 0.3: the equal-size and the ragged loop of
    icp_point_to_point against oracle.icp (the C oracle's nearest neighbours) -- transforms to 1e-4, fitness / rmse to 1e-5.
    The oracle settles in a local minimum (not the true pose) at iteration 18, with |delta rmse| 5.6e-6 one iteration before
    and 0 at it, so both loops must take the same number of iterations; the ragged loop's state shows it (converged after 18
    calls, not after 17).  The equal-size loop reports no convergence flag: its agreement in T is the check there."""
    import torch

    from genpc_b200.reg_xyz import _icp_point_to_point_ragged, icp_point_to_point

    tgt = clusters(3, 900)
    src = (tgt[::2] @ rot([1, -2, 0.5], 2.75)).astype(F32)

    def nn(cur, target):
        d, i = oracle.nn_distance(cur[None], target[None])
        return d[0], i[0]

    To, fo, ro, its = OI.icp(src, tgt, 0.3, nn=nn)
    assert its == 18
    Te, fe, re = icp_point_to_point(torch.from_numpy(src).to(cuda)[None], torch.from_numpy(tgt).to(cuda)[None], 0.3)
    assert np.abs(Te[0].cpu().numpy() - To).max() <= 1e-4
    assert abs(float(fe[0]) - fo) <= 1e-5 and abs(float(re[0]) - ro) <= 1e-5
    sp = np.full((1, len(src) + 13, 3), np.nan, F32)
    sp[0, :len(src)] = src
    tp = np.full((1, len(tgt) + 5, 3), np.nan, F32)
    tp[0, :len(tgt)] = tgt
    s, t = torch.from_numpy(sp).to(cuda), torch.from_numpy(tp).to(cuda)
    ls, lt = torch.tensor([len(src)], device=cuda), torch.tensor([len(tgt)], device=cuda)
    for max_it, converged in ((30, 1.0), (its - 1, 1.0), (its - 2, 0.0)):   # max_it + 1 calls at most
        T, st = _icp_point_to_point_ragged(s, t, 0.3, None, max_it, 1e-6, 1e-6, ls, lt)
        assert float(st[0, 2]) == converged, (max_it, st)
    T, st = _icp_point_to_point_ragged(s, t, 0.3, None, 30, 1e-6, 1e-6, ls, lt)
    assert np.abs(T[0].cpu().numpy() - To).max() <= 1e-4
    assert abs(float(st[0, 0]) - fo) <= 1e-5 and abs(float(st[0, 1]) - ro) <= 1e-5
