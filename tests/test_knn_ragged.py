"""Ragged k-NN batches: clouds with their own point counts in one launch (genpc_knn_mean_distance_ragged,
knn_mean_distance(..., lengths=), remove_statistical_outlier(..., lengths=)).

CPU: argument errors of the C entry, host-side checks of the lengths.
GPU: every cloud bit for bit its solo call and the oracle (k 1, 7, 20, 32; lengths around k, the 2048-point tile edge and the
stride; random, lattice and shape clouds); padding never read and written as -1; the batch forms against each other with one
kernel launch; the outlier masks against the oracle; no host synchronisation; the single-cloud mask against the parent's
formula; a dataset-sized batch."""
import ctypes

import numpy as np
import pytest

import oracle
from util import lattice_cloud, rand_cloud, shape_cloud


# ---- CPU ---------------------------------------------------------------------------------------------------------------

def test_ragged_knn_entry_rejects_bad_arguments_without_a_device():
    """NULL pointers, B outside [1, 65535], n < 0, k outside [1, 32]: GENPC_ERR_SHAPE before any CUDA call."""
    from genpc_b200 import _lib

    L = _lib.lib()
    buf = (ctypes.c_int * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)   # never dereferenced: the checks come first

    def knn(xyz=p, ln=p, B=2, n=8, k=4, out=p):
        return L.genpc_knn_mean_distance_ragged(xyz, ln, B, n, k, 1, out, None)

    assert knn(xyz=None) == -1 and knn(ln=None) == -1 and knn(out=None) == -1
    for B in (0, -1, 65536):
        assert knn(B=B) == -1, B
    assert knn(n=-1) == -1
    for k in (0, 33):
        assert knn(k=k) == -1, k
    assert knn(n=0) == 0   # nothing to do: nothing queued


def test_knn_lengths_are_checked_on_the_host():
    import torch

    from genpc_b200 import _lib
    from genpc_b200.reg_xyz import knn_mean_distance, remove_statistical_outlier

    xyz = torch.zeros(3, 10, 3)
    for bad in (torch.tensor([1.0, 2.0, 3.0]), torch.tensor([True, False, True]), torch.tensor([1, 2]),
                torch.tensor([[1, 2, 3]]), torch.tensor([1, 2, 3], device="meta"), [1, 2, 3]):
        with pytest.raises(_lib.GenpcError, match="len"):
            knn_mean_distance(xyz, 20, True, bad)
        with pytest.raises(_lib.GenpcError, match="len"):
            remove_statistical_outlier(xyz, 20, 2.5, bad)
    with pytest.raises(_lib.GenpcError, match="len"):   # one cloud has no lengths
        knn_mean_distance(xyz[0], 20, True, torch.tensor([10]))
    with pytest.raises(_lib.GenpcError, match="len"):
        remove_statistical_outlier(xyz[0], 20, 2.5, torch.tensor([10]))
    with pytest.raises(_lib.GenpcError, match="CPU"):   # well-formed lengths pass on to the no-CPU-fallback check
        knn_mean_distance(xyz, 20, True, torch.tensor([10, 0, 4]))


# ---- GPU ---------------------------------------------------------------------------------------------------------------

def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


def clouds(kind, seed, B, N):
    return {"rand": lambda: rand_cloud(seed, B, N), "lattice": lambda: lattice_cloud(seed, B, N, side=9),
            "shape": lambda: shape_cloud(seed, B, N)}[kind]()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 7, 20, 32])
def test_every_cloud_is_its_solo_call_and_the_oracle(cuda, k):
    """Cloud b of a ragged batch: rows j < len[b] bit for bit knn_mean_distance on x[b, :len[b]] alone and the oracle, rows past
    it -1.  The rows past a length hold points of the same kind (a kernel that read them would find nearer neighbours)."""
    import torch

    from genpc_b200.reg_xyz import knn_mean_distance

    S = 4101
    lens = sorted({0, 1, 2, k - 1, k, k + 1, 2047, 2048, 2049, 4097, S})
    for kind in ("rand", "lattice", "shape"):
        x = clouds(kind, 10 * k + len(kind), len(lens), S)
        t = torch.from_numpy(x).to(cuda)
        ln = torch.tensor(lens, dtype=torch.int32, device=cuda)
        for inc in (True, False):
            got = knn_mean_distance(t, k, inc, ln).cpu().numpy()
            for b, n in enumerate(lens):
                solo = knn_mean_distance(t[b, :n], k, inc).cpu().numpy()
                exp = oracle.knn_mean_distance(x[b, :n], k, inc)
                assert np.array_equal(bits(got[b, :n]), bits(solo)), (kind, inc, n)
                assert np.array_equal(bits(got[b, :n]), bits(exp)), (kind, inc, n)
                assert (got[b, n:] == -1).all(), (kind, inc, n)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [7, 20])
def test_padding_is_never_read(cuda, k):
    """Padding of NaN, +1e30 or -1e30 gives the bits of zero padding; padding rows are exactly -1."""
    import torch

    from genpc_b200.reg_xyz import knn_mean_distance

    lens = [0, 1, 31, 32, 33, 2048, 2049, 3000]
    S = 3000
    x = shape_cloud(7, len(lens), S)
    ln = torch.tensor(lens, dtype=torch.int32, device=cuda)
    runs = {}
    for fill in (0.0, float("nan"), 1e30, -1e30):
        y = x.copy()
        for b, n in enumerate(lens):
            y[b, n:] = fill
        t = torch.from_numpy(y).to(cuda)
        runs[fill] = [knn_mean_distance(t, k, inc, ln).cpu().numpy() for inc in (True, False)]
    for fill, outs in runs.items():
        for got, ref in zip(outs, runs[0.0]):
            assert np.array_equal(bits(got), bits(ref)), fill
            for b, n in enumerate(lens):
                assert np.array_equal(bits(got[b, n:]), bits(np.full(S - n, -1.0, np.float32))), (fill, n)


@pytest.mark.gpu
def test_batch_forms_agree_and_launch_once(cuda):
    """[B,N,3] without lengths, with every length at the stride, and B solo calls: the same bits.  Each batched call launches
    knn_mean_kernel<k> once, on a (query blocks, B) grid; the single-cloud entry keeps its 1-D grid (one profiler session)."""
    import torch

    from genpc_b200.reg_xyz import knn_mean_distance
    from test_dispatch_paths import launched_kernels

    B, N, k = 5, 2500, 20
    t = torch.from_numpy(shape_cloud(3, B, N)).to(cuda)
    full = torch.full((B,), N, dtype=torch.int64, device=cuda)
    solo = np.stack([knn_mean_distance(t[b], k).cpu().numpy() for b in range(B)])
    got, ks = launched_kernels(lambda: [knn_mean_distance(t, k, True, None).cpu().numpy(),
                                        knn_mean_distance(t, k, True, full).cpu().numpy(),
                                        knn_mean_distance(t[0], k).cpu().numpy()])
    assert np.array_equal(bits(got[0]), bits(solo)) and np.array_equal(bits(got[1]), bits(solo))
    assert np.array_equal(bits(got[2]), bits(solo[0]))
    gx = (N * 4 + 127) // 128
    assert [g for key, g, _ in ks if key == f"genpc::knn_mean_kernel<{k}>"] == [(gx, B, 1), (gx, B, 1), (gx, 1, 1)], ks


@pytest.mark.gpu
@pytest.mark.parametrize("r", [1.5, 2.5])
def test_batched_masks_match_the_oracle(cuda, r):
    """Per cloud, the batched mask is oracle.statistical_outlier_mask over the cloud's own points; padding is False.  Clouds of
    0 and 1 point take the nv <= 1 paths, a 2-point cloud the smallest nv > 1."""
    import torch

    from genpc_b200.reg_xyz import remove_statistical_outlier

    lens = [0, 1, 2, 3, 21, 500, 2049, 3500]
    S = 3500
    x = shape_cloud(11, len(lens), S)
    x[:, ::97] *= 1.6   # a few points off the surface, so that the threshold removes some
    t = torch.from_numpy(x).to(cuda)
    got = remove_statistical_outlier(t, 20, r, torch.tensor(lens, device=cuda)).cpu().numpy()
    assert got.dtype == bool and got.shape == (len(lens), S)
    for b, n in enumerate(lens):
        exp = oracle.statistical_outlier_mask(oracle.knn_mean_distance(x[b, :n], 20, True), r)
        assert np.array_equal(got[b, :n], exp), n
        assert not got[b, n:].any(), n
    assert not got[1, 0]   # one point: no neighbour but itself, mean 0 -> dropped
    assert 0 < got[-1].sum() < S


@pytest.mark.gpu
def test_outlier_filter_does_not_synchronise(cuda):
    import torch

    from genpc_b200.reg_xyz import remove_statistical_outlier

    t = torch.from_numpy(shape_cloud(5, 3, 3000)).to(cuda)
    ln = torch.tensor([3000, 17, 1200], dtype=torch.int32, device=cuda)
    remove_statistical_outlier(t[0], 20, 2.5), remove_statistical_outlier(t, 20, 1.5, ln)   # warm-up: module load
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        a = remove_statistical_outlier(t[0], 20, 2.5)
        b = remove_statistical_outlier(t, 20, 1.5, ln)
        c = remove_statistical_outlier(t, 20, 1.5)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert a.shape == (3000,) and b.shape == c.shape == (3, 3000)


def parent_mask(md, std_ratio):
    """remove_statistical_outlier's threshold as it read before batches existed (boolean indexing, host-side nv)."""
    import torch

    md = md.double()
    nv = int((md >= 0).sum())
    if nv == 0:
        return torch.zeros_like(md, dtype=torch.bool)
    pos = md > 0
    mu = md[pos].sum() / nv
    sd = torch.sqrt(((md[pos] - mu) ** 2).sum() / (nv - 1)) if nv > 1 else torch.zeros((), dtype=torch.float64, device=md.device)
    return pos & (md < mu + std_ratio * sd)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 7, 300, 5000, 20000, 4099, 2048])
def test_single_cloud_mask_equals_the_parent_formula(cuda, n):
    """The seeded clouds of tests/test_reg_xyz.py::test_knn_mean_distance_gpu_bit_exact: the masked float64 reduction gives
    the parent's mask (its sums ran in another order)."""
    import torch

    from genpc_b200.reg_xyz import knn_mean_distance, remove_statistical_outlier

    for x in (rand_cloud(n, 1, n)[0], lattice_cloud(n + 1, 1, n, side=9)[0], shape_cloud(n + 2, 1, n)[0]):
        t = torch.from_numpy(x).to(cuda)
        for r in (1.5, 2.5):
            assert torch.equal(remove_statistical_outlier(t, 20, r), parent_mask(knn_mean_distance(t, 20), r))


@pytest.mark.gpu
def test_dataset_sized_batch(cuda):
    """110 clouds of 300-20 000 points in one call: every cloud's means and mask equal its solo call; three clouds (the
    smallest, the largest, one between) also equal the oracle."""
    import torch

    from genpc_b200.optim_registration.diff_obj_pose import pad_clouds
    from genpc_b200.reg_xyz import knn_mean_distance, remove_statistical_outlier
    from genpc_b200.synthetic import superquadric

    rng = np.random.default_rng(0)
    sizes = [300, 20000] + [int(v) for v in rng.integers(300, 20001, 108)]
    xs = [superquadric(i, n) for i, n in enumerate(sizes)]
    pad, ln = pad_clouds([torch.from_numpy(x).to(cuda) for x in xs])
    md = knn_mean_distance(pad, 20, True, ln).cpu().numpy()
    keep = remove_statistical_outlier(pad, 20, 2.5, ln).cpu().numpy()
    for b, x in enumerate(xs):
        t = pad[b, :len(x)]
        assert np.array_equal(bits(md[b, :len(x)]), bits(knn_mean_distance(t, 20).cpu().numpy())), b
        assert np.array_equal(keep[b, :len(x)], remove_statistical_outlier(t, 20, 2.5).cpu().numpy()), b
        assert (md[b, len(x):] == -1).all() and not keep[b, len(x):].any(), b
    for b in (0, 1, 2):
        assert np.array_equal(bits(md[b, :len(xs[b])]), bits(oracle.knn_mean_distance(xs[b], 20, True))), b
