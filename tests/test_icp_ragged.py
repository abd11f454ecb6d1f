"""Ragged ICP batches: candidates with their own source / target point counts in one loop (genpc_icp_step_ragged,
icp_point_to_point(..., source_lengths=, target_lengths=), coarse_scale_sweep_batch).

CPU: argument errors of the C entry, host-side checks of the lengths, GENPC_ICP_TORCH=1 refusing lengths.
GPU: every candidate bit for bit its solo run on its sliced clouds (lengths 0, 1, 2, 3, odd sizes and the stride; different
convergence iterations; no inliers); padding never read; lengths at the strides against the equal-size loop; the oracle's
ICP; the dataset sweep against the per-object sweep."""
import ctypes
import math

import numpy as np
import pytest

import oracle
from oracle import icp as OI


# ---- CPU ---------------------------------------------------------------------------------------------------------------

def test_ragged_icp_entry_rejects_bad_arguments_without_a_device():
    """NULL source / length pointers, only one of dist / idx, Kt not in {1, K}, sizes <= 0: GENPC_ERR_SHAPE before any CUDA
    call."""
    from genpc_b200 import _lib

    L = _lib.lib()
    buf = (ctypes.c_int * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)   # never dereferenced: the checks come first

    def step(source=p, dist=p, idx=p, src_len=p, tgt_len=p, scan_len=p, K=2, Ns=8, Kt=2, Nt=8):
        return L.genpc_icp_step_ragged(source, p, p, dist, idx, src_len, tgt_len, scan_len, p, p, K, Ns, Kt, Nt, 0.01, 1e-6,
                                       1e-6, 1, None)

    assert step(source=None) == -1
    assert step(src_len=None) == -1 and step(tgt_len=None) == -1 and step(scan_len=None) == -1
    assert step(dist=None) == -1 and step(idx=None) == -1
    assert step(Kt=3) == -1 and step(K=3, Kt=2) == -1
    for bad in (dict(K=0, Kt=1), dict(K=-1, Kt=1), dict(Ns=0), dict(Ns=-4), dict(Nt=0), dict(Nt=-1)):
        assert step(**bad) == -1, bad


def test_icp_lengths_are_checked_on_the_host():
    import torch

    from genpc_b200 import _lib
    from genpc_b200.reg_xyz import _candidate_lengths, chamfer_partial_l1_batched, icp_point_to_point

    src, tgt = torch.zeros(3, 10, 3), torch.zeros(3, 7, 3)
    l1, l2 = _candidate_lengths(src, tgt, torch.tensor([10, 0, 4]), None)
    assert l1.dtype == l2.dtype == torch.int32 and l1.tolist() == [10, 0, 4] and l2.tolist() == [7, 7, 7]
    l1, l2 = _candidate_lengths(src, tgt[:1], None, torch.tensor([5]))   # a shared target's length goes with it
    assert l1.tolist() == [10, 10, 10] and l2.tolist() == [5, 5, 5]
    for bad in (torch.tensor([1.0, 2.0, 3.0]), torch.tensor([True, False, True]), torch.tensor([1, 2]),
                torch.tensor([[1, 2, 3]]), torch.tensor([1, 2, 3], device="meta"), [1, 2, 3]):
        for kw in (dict(source_lengths=bad), dict(target_lengths=bad)):
            with pytest.raises(_lib.GenpcError, match="len"):
                icp_point_to_point(src, tgt, 0.05, **kw)
        with pytest.raises(_lib.GenpcError, match="len"):
            chamfer_partial_l1_batched(src, tgt, 0.5, bad)


def test_icp_torch_formulation_refuses_lengths(monkeypatch):
    import torch

    from genpc_b200 import _lib
    from genpc_b200.reg_xyz import icp_point_to_point

    monkeypatch.setenv("GENPC_ICP_TORCH", "1")
    src, tgt = torch.zeros(2, 10, 3), torch.zeros(2, 7, 3)
    for kw in (dict(source_lengths=torch.tensor([10, 4])), dict(target_lengths=torch.tensor([7, 7]))):
        with pytest.raises(_lib.GenpcError, match="GENPC_ICP_TORCH"):
            icp_point_to_point(src, tgt, 0.05, **kw)


# ---- GPU ---------------------------------------------------------------------------------------------------------------

def candidates(sizes, seed=5):
    """(source, target) numpy clouds per candidate: rotated / shifted / slightly scaled subsets of one superquadric, rotation
    growing with k so that candidates converge at different iterations; sizes = [(n_source, n_target)]."""
    from genpc_b200.synthetic import superquadric

    base = superquadric(9, 4000)
    rng = np.random.default_rng(seed)
    out = []
    for k, (ns, nt) in enumerate(sizes):
        ang = 0.015 * (k % 7 + 1)
        R = np.array([[math.cos(ang), -math.sin(ang), 0], [math.sin(ang), math.cos(ang), 0], [0, 0, 1.0]], np.float32)
        t = ((rng.random(3) - 0.5) * 0.04).astype(np.float32)
        tgt = base[k % 5::5][:nt].copy()
        src = ((base[k % 3::3][:ns] - t) @ R * np.float32(1.0 + 0.01 * (k % 5 - 2))).astype(np.float32)
        out.append((src, tgt))
    return out


def pad(clouds, stride, fill=0.0):
    out = np.full((len(clouds), stride, 3), fill, np.float32)
    for i, c in enumerate(clouds):
        out[i, :len(c)] = c
    return out


def run(src, tgt, ls, lt, dev):
    """_icp_point_to_point_ragged on numpy inputs -> (T, state) as numpy."""
    import torch

    from genpc_b200.reg_xyz import _icp_point_to_point_ragged

    T, st = _icp_point_to_point_ragged(torch.from_numpy(src).to(dev), torch.from_numpy(tgt).to(dev), 0.075, None, 30, 1e-6,
                                       1e-6, torch.tensor(ls, device=dev), torch.tensor(lt, device=dev))
    return T.cpu().numpy(), st.cpu().numpy()


SIZES = [(1, 600), (2, 600), (3, 600), (37, 301), (257, 611), (611, 1), (700, 700), (699, 97), (450, 2), (700, 3)]
NS, NT = 700, 700


@pytest.mark.gpu
def test_every_candidate_equals_its_solo_run(cuda):
    """Each candidate of a ragged batch: T, fitness, rmse and converged bit for bit its run alone on its sliced clouds (the
    calls counter may differ: a batch runs until its slowest candidate converges).  Lengths 0 leave T at its start with
    fitness 0; a far-away candidate has no inliers and stays at the identity."""
    cands = candidates(SIZES)
    cands[8] = (cands[8][0] + np.float32(5.0), cands[8][1])         # far away: no inliers
    srcs, tgts = [c[0] for c in cands], [c[1] for c in cands]
    ls, lt = [len(s) for s in srcs], [len(t) for t in tgts]
    ls += [0, 300]
    lt += [500, 0]
    srcs += [np.zeros((0, 3), np.float32), srcs[4][:300]]
    tgts += [tgts[4][:500], np.zeros((0, 3), np.float32)]
    T, st = run(pad(srcs, NS), pad(tgts, NT), ls, lt, cuda)
    iters = set()
    for k, (s, t) in enumerate(zip(srcs, tgts)):
        if len(s) == 0 or len(t) == 0:
            assert np.array_equal(T[k], np.eye(4, dtype=np.float32)) and st[k, 0] == 0 and st[k, 1] == 0, k
            continue
        T1, st1 = run(s[None], t[None], [len(s)], [len(t)], cuda)
        assert np.array_equal(T[k].view(np.int32), T1[0].view(np.int32)), (k, np.abs(T[k] - T1[0]).max())
        assert np.array_equal(st[k, :3].view(np.int32), st1[0, :3].view(np.int32)), (k, st[k], st1[0])
        iters.add(int(st1[0, 3]))
    assert np.array_equal(T[8], np.eye(4, dtype=np.float32)) and st[8, 0] == 0
    assert st[6, 0] > 0.9 and st[4, 0] > 0.9
    assert len(iters) >= 2, iters   # candidates converge at different iterations


@pytest.mark.gpu
def test_padding_is_never_read(cuda):
    cands = candidates(SIZES[3:8])
    srcs, tgts = [c[0] for c in cands], [c[1] for c in cands]
    ls, lt = [len(s) for s in srcs], [len(t) for t in tgts]
    ref = run(pad(srcs, NS + 5), pad(tgts, NT + 3), ls, lt, cuda)
    for fill in (np.nan, 1e30, -1e30):
        got = run(pad(srcs, NS + 5, fill), pad(tgts, NT + 3, fill), ls, lt, cuda)
        for a, b in zip(got, ref):
            assert np.array_equal(a.view(np.int32), b.view(np.int32)), fill


@pytest.mark.gpu
@pytest.mark.parametrize("shared", [True, False])
def test_lengths_at_the_strides_match_the_equal_size_loop(cuda, shared):
    """Every length at its stride: the equal-size icp_point_to_point within the tolerance of its torch A/B check (the clouds
    are transformed with another rounding), for a shared [1,Nt,3] and a per-candidate target."""
    import torch

    from genpc_b200.reg_xyz import icp_point_to_point

    cands = candidates([(NS, NT)] * 7)
    src = torch.from_numpy(np.stack([c[0] for c in cands])).to(cuda)
    src[-1] += 5.0                                                   # no inliers
    tgt = torch.from_numpy(cands[0][1] if shared else np.stack([c[1] for c in cands])).to(cuda)
    tgt = tgt[None] if shared else tgt
    Te, fe, re = icp_point_to_point(src, tgt, 0.075)
    lt = torch.tensor([NT] if shared else [NT] * 7, device=cuda)
    Tr, fr, rr = icp_point_to_point(src, tgt, 0.075, source_lengths=torch.full((7,), NS, device=cuda), target_lengths=lt)
    assert torch.allclose(Tr, Te, atol=1e-4), (Tr - Te).abs().max()
    assert torch.allclose(fr, fe, atol=1e-5) and torch.allclose(rr, re, atol=1e-5)
    assert torch.equal(Tr[-1], torch.eye(4, device=cuda)) and float(fr[-1]) == 0.0
    assert float(fr[:-1].min()) > 0.9


@pytest.mark.gpu
def test_every_candidate_agrees_with_the_oracle(cuda):
    """Each candidate against oracle.icp on its sliced clouds (the C oracle's nearest neighbours).  Targets of one or two points
    are left out: there every rotation is optimal, and Horn's form and the oracle's SVD pick different ones."""
    cands = [c for c in candidates(SIZES) if len(c[1]) >= 3]
    srcs, tgts = [c[0] for c in cands], [c[1] for c in cands]
    ls, lt = [len(s) for s in srcs], [len(t) for t in tgts]
    T, st = run(pad(srcs, NS), pad(tgts, NT), ls, lt, cuda)

    def nn(cur, target):
        d, i = oracle.nn_distance(cur[None], target[None])
        return d[0], i[0]

    for k, (s, t) in enumerate(zip(srcs, tgts)):
        To, fo, ro, _ = OI.icp(s, t, 0.075, nn=nn)
        assert np.abs(T[k] - To).max() <= 1e-4, (k, np.abs(T[k] - To).max())
        assert abs(st[k, 0] - fo) <= 1e-5 and abs(st[k, 1] - ro) <= 1e-5, (k, st[k], fo, ro)


def sweep_objects(n, seed=11):
    """n seeded (scan, generated shape) pairs of different sizes, the scan a scaled, rigidly moved partial view."""
    from genpc_b200.synthetic import partial_view, rigid_perturb, superquadric

    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        nt, ns = int(rng.integers(300, 2601)), int(rng.integers(300, 1401))
        comp = superquadric(seed + i, nt)
        part, _ = rigid_perturb(partial_view(comp, seed + i, ns), seed + i, max_rot_deg=8.0, max_t=0.03,
                                scale_range=(0.7, 0.9))
        out.append((part.astype(np.float32), comp.astype(np.float32)))
    return out


@pytest.mark.gpu
def test_dataset_sweep_matches_the_per_object_sweep(cuda):
    """coarse_scale_sweep_batch over 12 objects against coarse_scale_sweep per object: the same best scale, the loss within
    1e-5 relative, the transform within 1e-4; and each object's result is bit for bit the same alone or in the batch."""
    import torch

    from genpc_b200.reg_xyz import coarse_scale_sweep, coarse_scale_sweep_batch

    objs = [(torch.from_numpy(s).to(cuda), torch.from_numpy(t).to(cuda)) for s, t in sweep_objects(12)]
    scales = np.linspace(1.5, 0.8, 11)
    batch = coarse_scale_sweep_batch([s for s, _ in objs], [t for _, t in objs], scales)
    assert len(batch) == len(objs)
    for i, (s, t) in enumerate(objs):
        ref = coarse_scale_sweep(s, t, scales, 0.075, 0.5)
        got = batch[i]
        assert got["best_scale"] == ref["best_scale"], (i, got["best_scale"], ref["best_scale"])
        assert abs(got["coarse_loss"] - ref["coarse_loss"]) <= 1e-5 * abs(ref["coarse_loss"]), (i, got, ref)
        assert torch.allclose(got["coarse_transformation"], ref["coarse_transformation"], atol=1e-4), i
        alone = coarse_scale_sweep_batch([s], [t], scales)[0]
        assert alone["best_scale"] == got["best_scale"], i
        assert torch.equal(alone["coarse_transformation"], got["coarse_transformation"]), i
