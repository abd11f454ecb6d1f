"""Ragged Chamfer batches: cloud pairs of different sizes in one call (genpc_chamfer_forward_ragged,
genpc_chamfer_loss_backward_ragged, chamfer_3DDist()(a, b, lengths1, lengths2), Completionloss.get_loss(gen, gt, gen_lengths,
gt_lengths), GraphedLossStep with lengths).

CPU: argument errors of the C entries, host-side checks of the lengths, EMD refusing lengths, pad_clouds feeding the lengths.
GPU: every pair bit for bit the oracle on its sliced clouds (0 / -1 for rows without a neighbour); padding never read; lengths
at the strides equal the equal-size call; the fused loss and its gradients against float64 per-pair means; autograd against
the oracle's backward; armed-workspace reuse across ragged and equal-size calls; CUDA-graph replay with new lengths."""
import ctypes

import numpy as np
import pytest

import oracle
from util import lattice_cloud, rand_cloud, shape_cloud


# ---- CPU ---------------------------------------------------------------------------------------------------------------

def test_ragged_entries_reject_bad_arguments_without_a_device():
    """NULL lengths / negative sizes: GENPC_ERR_SHAPE; a missing or too small workspace (packed words or loss partials):
    GENPC_ERR_WORKSPACE; an item grid beyond 2^31: GENPC_ERR_RANGE -- all before any CUDA call."""
    from genpc_b200 import _lib

    L = _lib.lib()
    buf = (ctypes.c_int * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)   # never dereferenced: the checks come first

    def fwd(l1, l2, B, N, M, ws=None, nbytes=0, fuse=None):
        return L.genpc_chamfer_forward_ragged(p, p, l1, l2, p, p, p, p, B, N, M, ws, nbytes, fuse, None)

    assert fwd(None, p, 2, 8, 8) == -1
    assert fwd(p, None, 2, 8, 8) == -1
    assert fwd(p, p, -1, 8, 8) == -1 and fwd(p, p, 2, -8, 8) == -1 and fwd(p, p, 2, 8, -1) == -1
    assert fwd(p, p, 2, 8, 8) == -2
    assert fwd(p, p, 2, 8, 8, p, L.genpc_chamfer_workspace_bytes(2, 8, 8) - 1) == -2
    fuse = _lib.ChamferFuse(0, 1, 0.5, 0.5, ctypes.cast(buf, ctypes.c_void_p).value, None, 0, None, None)
    assert fwd(p, p, 2, 8, 8, p, 1 << 20, ctypes.byref(fuse)) == -2
    assert fwd(p, p, 200000, 1000000, 1000000, p, 1 << 62) == -3

    def bwd(l1, l2, B, N, M):
        return L.genpc_chamfer_loss_backward_ragged(p, p, l1, l2, p, p, p, p, p, 1, 0.5, 0.5, p, p, B, N, M, None)

    assert bwd(None, p, 2, 8, 8) == -1 and bwd(p, None, 2, 8, 8) == -1
    assert bwd(p, p, 2, -8, 8) == -1


def test_python_layer_checks_lengths_on_the_host():
    import torch

    from genpc_b200 import _lib, chamfer_3D
    from genpc_b200.loss_functions import chamfer_3DDist

    a, b = torch.zeros(3, 10, 3), torch.zeros(3, 7, 3)
    ok = torch.tensor([10, 0, 4])
    l1, l2 = chamfer_3D.lengths(a, b, ok, None)
    assert l1.dtype == torch.int32 and l1.tolist() == [10, 0, 4] and l2.tolist() == [7, 7, 7]
    assert chamfer_3D.lengths(a, b, None, None) is None
    for bad in (torch.tensor([1.0, 2.0, 3.0]), torch.tensor([True, False, True]), torch.tensor([1, 2]),
                torch.tensor([[1, 2, 3]]), torch.tensor([1, 2, 3], device="meta"), [1, 2, 3]):
        with pytest.raises(_lib.GenpcError):
            chamfer_3DDist()(a, b, bad)
        with pytest.raises(_lib.GenpcError):
            chamfer_3DDist()(a, b, None, bad[:3] if isinstance(bad, list) else bad)


def test_emd_takes_no_lengths():
    import torch

    from genpc_b200.utils.loss_util import Completionloss

    x = torch.zeros(2, 256, 3)
    with pytest.raises(ValueError):
        Completionloss("emd").get_loss(x, x, torch.tensor([256, 100]))
    with pytest.raises(ValueError):
        Completionloss("emd").get_loss(x, x, None, torch.tensor([256, 100]))


def test_pad_clouds_feeds_the_lengths():
    import torch

    from genpc_b200 import chamfer_3D
    from genpc_b200.optim_registration.diff_obj_pose import pad_clouds

    rng = np.random.default_rng(3)
    c1 = [torch.from_numpy(rng.random((n, 3), dtype=np.float32)) for n in (5, 40, 1)]
    c2 = [torch.from_numpy(rng.random((n, 3), dtype=np.float32)) for n in (33, 2, 9)]
    x1, n1 = pad_clouds(c1)
    x2, n2 = pad_clouds(c2)
    l1, l2 = chamfer_3D.lengths(x1, x2, n1, n2)
    assert l1.tolist() == [5, 40, 1] and l2.tolist() == [33, 2, 9] and l1.dtype == l2.dtype == torch.int32
    for i, c in enumerate(c1):
        assert torch.equal(x1[i, :int(l1[i])], c)


# ---- GPU ---------------------------------------------------------------------------------------------------------------

def expected(a, b, l1, l2):
    """Per pair: the oracle on the sliced clouds; rows past a length, and every row of a pair whose other cloud is empty,
    0 / -1 (for an empty side the oracle zero-fills indices as 0, DESIGN section 3.1, so it is not asked)."""
    B, N, _ = a.shape
    M = b.shape[1]
    d1, d2 = np.zeros((B, N), np.float32), np.zeros((B, M), np.float32)
    i1, i2 = np.full((B, N), -1, np.int32), np.full((B, M), -1, np.int32)
    for k in range(B):
        n, m = int(l1[k]), int(l2[k])
        if n == 0 or m == 0:
            continue
        e = oracle.chamfer_forward(a[k:k + 1, :n], b[k:k + 1, :m])
        d1[k, :n], d2[k, :m], i1[k, :n], i2[k, :m] = e[0][0], e[1][0], e[2][0], e[3][0]
    return d1, d2, i1, i2


def run_ragged(a, b, l1, l2, dev):
    import torch

    from genpc_b200.loss_functions import chamfer_3DDist

    out = chamfer_3DDist()(torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev), torch.from_numpy(np.asarray(l1)).to(dev),
                           torch.from_numpy(np.asarray(l2)).to(dev))
    return [t.cpu().numpy() for t in out]


def assert_bits(got, exp, what):
    for g, e, name in zip(got, exp, ("dist1", "dist2", "idx1", "idx2")):
        assert g.dtype == e.dtype and np.array_equal(g.view(np.int32), e.view(np.int32)), \
            f"{what}: {name} differs in {(g.view(np.int32) != e.view(np.int32)).sum()} entries"


def lengths_for(rng, B, n):
    """Lengths for B pairs of stride n: 0, 1 and n among them, the rest random."""
    ln = rng.integers(0, n + 1, size=B)
    special = [0, 1, n, n, 1 if n > 1 else 0]
    ln[:min(B, len(special))] = special[:min(B, len(special))]
    return rng.permutation(ln).astype(np.int32)


# (moving points, fixed points) per pair as in test_registration_ragged
RAGGED_SIZES = [(37, 64), (300, 1100), (1201, 517), (2600, 1400), (950, 230), (2600, 1400)]


@pytest.mark.gpu
def test_mixed_pairs_bit_exact_vs_oracle(cuda):
    """Registration-sized pairs of test_registration_ragged.make_pairs, both orientations (N > M and N < M)."""
    from test_registration_ragged import make_pairs

    pairs = make_pairs(RAGGED_SIZES, seed0=40)
    N, M = max(c.shape[0] for c, _ in pairs), max(p.shape[0] for _, p in pairs)
    a, b = np.zeros((len(pairs), N, 3), np.float32), np.zeros((len(pairs), M, 3), np.float32)
    for k, (c, p) in enumerate(pairs):
        a[k, :len(c)], b[k, :len(p)] = c, p
    l1 = np.array([len(c) for c, _ in pairs], np.int32)
    l2 = np.array([len(p) for _, p in pairs], np.int32)
    assert_bits(run_ragged(a, b, l1, l2, cuda), expected(a, b, l1, l2), "N > M")
    assert_bits(run_ragged(b, a, l2, l1, cuda), expected(b, a, l2, l1), "N < M")


@pytest.mark.gpu
@pytest.mark.parametrize("N,M", [(1, 1), (31, 33), (33, 31), (513, 31), (31, 513), (513, 2049), (2049, 513), (2049, 2049)])
def test_strides_and_edge_lengths_bit_exact_vs_oracle(cuda, N, M):
    """Strides 1, 31, 33, 513, 2049 on either side; lengths 0, 1 and the stride on one side or both; random and lattice clouds
    (exact ties: the lowest index must win as in the pair alone)."""
    rng = np.random.default_rng(N * 7 + M)
    B = 7
    l1, l2 = lengths_for(rng, B, N), lengths_for(rng, B, M)
    l2[0], l1[0] = 0, N           # one pair with an empty second cloud, one with an empty first
    l1[1], l2[1] = 0, M
    for kind, (a, b) in (("rand", (rand_cloud(N + 1, B, N), rand_cloud(M + 2, B, M, 0.8, -0.2))),
                         ("lattice", (lattice_cloud(N + 3, B, N, side=4), lattice_cloud(M + 4, B, M, side=4)))):
        got = run_ragged(a, b, l1, l2, cuda)
        assert_bits(got, expected(a, b, l1, l2), f"{kind} {N}x{M} {l1.tolist()} {l2.tolist()}")


@pytest.mark.gpu
def test_padding_is_never_read(cuda):
    """NaN and +-inf in every padding row give the outputs of zero padding, bit for bit (forward, fused loss, gradients)."""
    import torch

    from genpc_b200.utils.loss_util import Completionloss

    rng = np.random.default_rng(11)
    B, N, M = 6, 700, 1300
    l1, l2 = lengths_for(rng, B, N), lengths_for(rng, B, M)
    a0, b0 = shape_cloud(1, B, N), shape_cloud(2, B, M)
    res = []
    for pad in (0.0, float("nan"), float("inf"), float("-inf")):
        a, b = a0.copy(), b0.copy()
        for k in range(B):
            a[k, l1[k]:], b[k, l2[k]:] = pad, pad
        out = run_ragged(a, b, l1, l2, cuda)
        ta = torch.from_numpy(a).to(cuda).requires_grad_(True)
        tb = torch.from_numpy(b).to(cuda).requires_grad_(True)
        loss = Completionloss("cd_l1").get_loss(ta, tb, torch.from_numpy(l1).to(cuda), torch.from_numpy(l2).to(cuda))
        loss.backward()
        res.append(out + [loss.detach().cpu().numpy(), ta.grad.cpu().numpy(), tb.grad.cpu().numpy()])
    for r in res[1:]:
        for x, y in zip(r[:5], res[0][:5]):
            assert np.array_equal(x.view(np.int32), y.view(np.int32))
        for x, y in zip(r[5:], res[0][5:]):   # (the gradients' atomics add in any order)
            assert np.abs(x - y).max() <= 1e-6 * np.abs(y).max()
    assert_bits(res[0][:4], expected(a0, b0, l1, l2), "zero padding")


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,M", [(3, 700, 1500), (32, 2048, 16384)])
def test_lengths_at_the_strides_equal_the_equal_size_call(cuda, B, N, M):
    """dist / idx bit-identical to the unragged call (the second shape takes the pruned scan unragged, the exhaustive one
    ragged); the fused loss within 1e-6 relative (summation order); the loss gradients' terms are bit-identical (graddist =
    w / (B * len) with len = the stride is the unragged w / (B * N)), their sums within 1e-6 (the atomics add in any order)."""
    import torch

    from genpc_b200.loss_functions import chamfer_3DDist
    from genpc_b200.utils.loss_util import Completionloss

    a = torch.from_numpy(shape_cloud(5, B, N)).to(cuda)
    b = torch.from_numpy(rand_cloud(6, B, M, 0.9, -0.45)).to(cuda)
    full1 = torch.full((B,), N, dtype=torch.int64, device=cuda)
    full2 = torch.full((B,), M, dtype=torch.int32, device=cuda)
    plain = chamfer_3DDist()(a, b)
    ragged = chamfer_3DDist()(a, b, full1, full2)
    for x, y in zip(plain, ragged):
        assert torch.equal(x, y)
    for form in ("cd_l1", "cd_l2"):
        cl = Completionloss(form)
        for fn in (cl.get_loss, cl.partial_matching):
            res = []
            for lens in ((None, None), (full1, full2)):
                ta, tb = a.clone().requires_grad_(True), b.clone().requires_grad_(True)
                loss = fn(ta, tb, *lens)
                loss.backward()
                res.append((float(loss.detach()), ta.grad, tb.grad))
            assert abs(res[0][0] - res[1][0]) <= 1e-6 * abs(res[0][0]), (form, res[0][0], res[1][0])
            for k in (1, 2):
                assert (res[0][k] - res[1][k]).abs().max() <= 1e-6 * res[0][k].abs().max(), form


def loss_oracle(a, b, l1, l2, use_sqrt, w1, w2):
    """float64 per-pair means over the oracle's distances; float64 gradients of them (oracle.chamfer_backward per pair with
    graddist = w / (B * len) (* 0.5 / sqrt d))."""
    B = a.shape[0]
    f = np.sqrt if use_sqrt else (lambda d: d)
    loss = 0.0
    g1, g2 = np.zeros(a.shape, np.float64), np.zeros(b.shape, np.float64)
    for k in range(B):
        n, m = int(l1[k]), int(l2[k])
        if n == 0 or m == 0:
            continue
        d1, d2, i1, i2 = oracle.chamfer_forward(a[k:k + 1, :n], b[k:k + 1, :m])
        loss += w1 * f(d1.astype(np.float64)).mean() / B + w2 * f(d2.astype(np.float64)).mean() / B
        s1 = np.full(d1.shape, w1 / (B * n)) * (0.5 / np.sqrt(d1.astype(np.float64)) if use_sqrt else 1.0)
        s2 = np.full(d2.shape, w2 / (B * m)) * (0.5 / np.sqrt(d2.astype(np.float64)) if use_sqrt else 1.0)
        e1, e2 = oracle.chamfer_backward(a[k:k + 1, :n], b[k:k + 1, :m], s1.astype(np.float32), s2.astype(np.float32), i1, i2)
        g1[k, :n], g2[k, :m] = e1[0], e2[0]
    return loss, g1, g2


@pytest.mark.gpu
def test_fused_loss_and_gradients_vs_float64_per_pair_means(cuda):
    """All four Chamfer forms, fused and literal torch (fused=False): loss within 1e-6, gradients within 1e-5 of the float64
    oracle; padding rows get exactly zero gradient; fused equals unfused within the same tolerances."""
    import torch

    from genpc_b200.utils.loss_util import Completionloss

    rng = np.random.default_rng(21)
    B, N, M = 9, 1600, 2600
    l1, l2 = lengths_for(rng, B, N), lengths_for(rng, B, M)
    a, b = shape_cloud(31, B, N), shape_cloud(32, B, M) * np.float32(1.1)
    forms = [("cd_l1", "get_loss", True, 0.5, 0.5), ("cd_l2", "get_loss", False, 1.0, 1.0),
             ("cd_l1", "chamfer_partial_l1", True, 1.0, 0.0), ("cd_l2", "chamfer_partial_l2", False, 1.0, 0.0)]
    for form, meth, use_sqrt, w1, w2 in forms:
        exp, e1, e2 = loss_oracle(a, b, l1, l2, use_sqrt, w1, w2)
        res = []
        for fused in (True, False):
            cl = Completionloss(form)
            cl.fused = fused
            ta = torch.from_numpy(a).to(cuda).requires_grad_(True)
            tb = torch.from_numpy(b).to(cuda).requires_grad_(True)
            loss = getattr(cl, meth)(ta, tb, torch.from_numpy(l1).to(cuda), torch.from_numpy(l2).to(cuda))
            loss.backward()
            g1, g2 = ta.grad.cpu().numpy(), tb.grad.cpu().numpy()
            assert abs(float(loss.detach()) - exp) <= 1e-6 * abs(exp), (form, meth, fused, float(loss.detach()), exp)
            for g, e in ((g1, e1), (g2, e2)):
                assert np.abs(g - e).max() <= 1e-5 * np.abs(e).max() + 1e-12, (form, meth, fused, np.abs(g - e).max())
            for k in range(B):
                assert not g1[k, l1[k]:].any() and not g2[k, l2[k]:].any(), (form, meth, fused, k)
            res.append((float(loss.detach()), g1, g2))
        assert abs(res[0][0] - res[1][0]) <= 1e-6 * abs(res[1][0])
        for k in (1, 2):
            assert np.abs(res[0][k] - res[1][k]).max() <= 1e-5 * np.abs(res[1][k]).max() + 1e-12


@pytest.mark.gpu
def test_autograd_through_chamfer_3DDist_with_lengths(cuda):
    """Random upstream gradients of dist1 / dist2 through the plain backward: each pair's gradients equal
    oracle.chamfer_backward on its sliced clouds within 1e-5; padding rows get zero."""
    import torch

    from genpc_b200.loss_functions import chamfer_3DDist

    rng = np.random.default_rng(5)
    B, N, M = 5, 900, 2100
    l1, l2 = lengths_for(rng, B, N), lengths_for(rng, B, M)
    a, b = shape_cloud(41, B, N), rand_cloud(42, B, M, 0.8, -0.4)
    g1 = rng.random((B, N), dtype=np.float32)
    g2 = rng.random((B, M), dtype=np.float32)
    ta = torch.from_numpy(a).to(cuda).requires_grad_(True)
    tb = torch.from_numpy(b).to(cuda).requires_grad_(True)
    d1, d2, _, _ = chamfer_3DDist()(ta, tb, torch.from_numpy(l1).to(cuda), torch.from_numpy(l2).to(cuda))
    ((d1 * torch.from_numpy(g1).to(cuda)).sum() + (d2 * torch.from_numpy(g2).to(cuda)).sum()).backward()
    ga, gb = ta.grad.cpu().numpy(), tb.grad.cpu().numpy()
    for k in range(B):
        n, m = int(l1[k]), int(l2[k])
        assert not ga[k, n:].any() and not gb[k, m:].any()
        if n == 0 or m == 0:
            assert not ga[k].any() and not gb[k].any()
            continue
        _, _, i1, i2 = oracle.chamfer_forward(a[k:k + 1, :n], b[k:k + 1, :m])
        e1, e2 = oracle.chamfer_backward(a[k:k + 1, :n], b[k:k + 1, :m], g1[k:k + 1, :n], g2[k:k + 1, :m], i1, i2)
        for g, e in ((ga[k, :n], e1[0]), (gb[k, :m], e2[0])):
            assert np.abs(g - e).max() <= 1e-5 * np.abs(e).max() + 1e-12, (k, np.abs(g - e).max())


@pytest.mark.gpu
def test_armed_workspace_reuse_across_ragged_and_equal_size_calls(cuda):
    """Ragged fused calls with changing lengths alternate with equal-size fused calls of the same (B, N, M) on one cached
    step workspace (left armed by each); the results equal those of fresh-workspace calls of the plain C entries."""
    import torch

    from genpc_b200 import _lib, chamfer_3D

    L = _lib.lib()
    rng = np.random.default_rng(8)
    for B, N, M in ((4, 1500, 900), (32, 2048, 16384)):
        for step in range(6):
            a = torch.from_numpy(shape_cloud(50 + step, B, N)).to(cuda)
            b = torch.from_numpy(rand_cloud(60 + step, B, M, 0.8, -0.4)).to(cuda)
            ragged = step % 2 == 0
            lens = chamfer_3D.lengths(a, b, torch.from_numpy(lengths_for(rng, B, N)).to(cuda),
                                      torch.from_numpy(lengths_for(rng, B, M)).to(cuda)) if ragged else None
            outs = [torch.empty(B, N, device=cuda), torch.empty(B, M, device=cuda),
                    torch.empty(B, N, dtype=torch.int32, device=cuda), torch.empty(B, M, dtype=torch.int32, device=cuda)]
            loss = torch.empty((), device=cuda)
            chamfer_3D.forward_fused(a, b, *outs, None, None, (loss, 1, 0.5, 0.5), lengths=lens)
            ref = [torch.empty_like(t) for t in outs]
            if ragged:
                chamfer_3D.forward_ragged(a, b, *ref, *lens)
            else:
                chamfer_3D.forward(a, b, *ref)
            for x, y in zip(outs, ref):
                assert torch.equal(x, y), (B, N, M, step)
            ws = chamfer_3D.step_workspace(a.device, B, N, M)
            assert ws.armed
            fresh = torch.empty((), device=cuda)
            fws = torch.zeros(L.genpc_chamfer_fuse_workspace_bytes(B, N, M), dtype=torch.uint8, device=cuda)
            pk = torch.empty(L.genpc_chamfer_workspace_bytes(B, N, M), dtype=torch.uint8, device=cuda)
            fuse = _lib.ChamferFuse(0, 1, 0.5, 0.5, fresh.data_ptr(), fws.data_ptr(), fws.numel(), None, None)
            args = (_lib.ptr(a), _lib.ptr(b))
            tail = (*[_lib.ptr(t) for t in ref], B, N, M, _lib.ptr(pk), pk.numel(), ctypes.byref(fuse), _lib.current_stream(cuda))
            rc = (L.genpc_chamfer_forward_ragged(*args, _lib.ptr(lens[0]), _lib.ptr(lens[1]), *tail) if ragged
                  else L.genpc_chamfer_forward_fused(*args, *tail))
            assert rc == 0
            assert torch.equal(loss, fresh), (B, N, M, step, float(loss), float(fresh))


@pytest.mark.gpu
def test_graph_replay_with_new_clouds_and_lengths(cuda):
    """A GraphedLossStep captured with lengths, replayed after writing new clouds and new lengths, equals the eager step."""
    import torch

    from genpc_b200.utils.loss_util import Completionloss, GraphedLossStep

    rng = np.random.default_rng(13)
    B, N, M = 8, 1800, 2400
    cl = Completionloss("cd_l1")

    def inputs(seed):
        return (torch.from_numpy(shape_cloud(seed, B, N)).to(cuda), torch.from_numpy(shape_cloud(seed + 1, B, M)).to(cuda),
                torch.from_numpy(lengths_for(rng, B, N)).to(cuda), torch.from_numpy(lengths_for(rng, B, M)).to(cuda))

    step = GraphedLossStep(cl, *inputs(70)[:2], gen_lengths=inputs(71)[2], gt_lengths=inputs(72)[3])
    for seed in (80, 90, 100):
        g, t, lg, lt = inputs(seed)
        loss, gg, gt = step(g, t, lg, lt)
        torch.cuda.synchronize()
        ta, tb = g.clone().requires_grad_(True), t.clone().requires_grad_(True)
        eager = cl.get_loss(ta, tb, lg, lt)
        eager.backward()
        assert torch.equal(loss, eager.detach()), seed
        for x, y in ((gg, ta.grad), (gt, tb.grad)):   # (the gradients' atomics add in any order)
            assert (x - y).abs().max() <= 1e-6 * y.abs().max(), seed
