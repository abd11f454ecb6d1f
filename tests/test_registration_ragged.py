"""Ragged registration batches: cloud pairs of different sizes in one run (genpc_register_run_ragged,
RegistrationBatch(complete_lengths=, partial_lengths=), RegistrationBatch.from_clouds).

CPU: padding, lengths and centres of from_clouds' helpers; the host-side argument checks of the C entry.
GPU: lengths equal to the strides reproduce the equal-size batch bit for bit (persistent and launch-per-iteration forms);
every pair of a ragged batch follows oracle/registration.py on that pair alone within 1e-5 and its solo RegistrationBatch
run within 1e-6; padding is never read; batches too large to be co-resident, split run() calls and problems above the
symmetric-path threshold take the single-launch kernels and agree."""
import ctypes

import numpy as np
import pytest

from oracle import registration as OR

# (moving points, fixed points) per pair; the last pair fills both strides
RAGGED_SIZES = [(37, 64), (300, 1100), (1201, 517), (2600, 1400), (950, 230), (2600, 1400)]


def make_pair(seed, nc, nr):
    from genpc_b200.synthetic import partial_view, rigid_perturb, superquadric

    comp = superquadric(seed, nc)
    part, _ = rigid_perturb(partial_view(comp, seed, nr), seed, max_rot_deg=20.0, max_t=0.05, scale_range=(0.7, 0.9))
    return comp, part


def make_pairs(sizes, seed0=500):
    return [make_pair(seed0 + i, nc, nr) for i, (nc, nr) in enumerate(sizes)]


def ragged_batch(cuda, pairs, starts, iters, pad=None):
    """RegistrationBatch.from_clouds on the pairs; pad: value written into the padded rows (None: the zeros of from_clouds)."""
    import torch

    from genpc_b200.optim_registration.diff_obj_pose import RegistrationBatch

    rb = RegistrationBatch.from_clouds([torch.from_numpy(c).to(cuda) for c, _ in pairs],
                                       [torch.from_numpy(p).to(cuda) for _, p in pairs], n_starts=starts, lr=0.01,
                                       max_iters=iters)
    if pad is not None:
        for i, (c, p) in enumerate(pairs):
            rb.complete[i, len(c):] = pad
            rb.partial[i, len(p):] = pad
    return rb


def result(rb):
    import torch

    torch.cuda.synchronize()
    return rb.params.cpu().numpy().copy(), rb.losses().cpu().numpy().copy()


# ---- CPU ---------------------------------------------------------------------------------------------------------------

def test_pad_clouds_lengths_and_centers_on_cpu():
    import torch

    from genpc_b200.optim_registration.diff_obj_pose import cloud_centers, pad_clouds

    rng = np.random.default_rng(0)
    clouds = [torch.from_numpy(rng.standard_normal((n, 3)).astype(np.float32)) for n in (5, 17, 1, 9)]
    padded, lengths = pad_clouds(clouds)
    assert padded.shape == (4, 17, 3) and padded.dtype == torch.float32
    assert lengths.dtype == torch.int32 and lengths.tolist() == [5, 17, 1, 9]
    for i, c in enumerate(clouds):
        assert torch.equal(padded[i, :len(c)], c)
        assert (padded[i, len(c):] == 0).all()
    centers = cloud_centers(padded, lengths)
    assert centers.shape == (4, 3)
    for i, c in enumerate(clouds):
        assert torch.equal(centers[i], c[None].mean(1)[0])          # the reduction a solo batch of that cloud makes
        assert torch.allclose(centers[i].double(), c.double().mean(0), rtol=0, atol=1e-6)
    assert torch.equal(cloud_centers(padded), padded.mean(1))        # no lengths: today's centre
    with pytest.raises(ValueError):
        pad_clouds([torch.zeros(4, 2)])
    with pytest.raises(ValueError):
        pad_clouds([])


def test_from_clouds_and_lengths_need_cuda_tensors():
    import torch

    from genpc_b200 import _lib
    from genpc_b200.optim_registration.diff_obj_pose import RegistrationBatch

    with pytest.raises(_lib.GenpcError):
        RegistrationBatch.from_clouds([torch.zeros(5, 3)], [torch.zeros(7, 3)])


def _ragged_call(L, len_ptr, S, n_starts, Nc, Nr):
    buf = (ctypes.c_int * 8)()
    p = ctypes.cast(buf, ctypes.c_void_p)   # never dereferenced: the checks come first
    ws = ctypes.create_string_buffer(16)
    return L.genpc_register_run_ragged(p, p, p, len_ptr, len_ptr, p, p, p, None, S, n_starts, Nc, Nr, 10, 0, 10, 0.01,
                                       0.002, 0.001, 1.0, 0.5, 3.0, ctypes.cast(ws, ctypes.c_void_p), 16, 1, None)


def test_ragged_entry_rejects_bad_arguments_without_a_device():
    """A null length pointer, S not a multiple of n_starts and Nc <= 0 give GENPC_ERR_SHAPE before any CUDA call."""
    from genpc_b200 import _lib

    L = _lib.lib()
    lens = (ctypes.c_int * 8)(*([16] * 8))
    lp = ctypes.cast(lens, ctypes.c_void_p)
    assert _ragged_call(L, None, 8, 4, 16, 16) == -1
    assert L.genpc_register_run_ragged(None, None, None, lp, None, None, None, None, None, 8, 4, 16, 16, 1, 0, 1, 0.01,
                                       0.002, 0.001, 1.0, 0.5, 3.0, None, 0, 1, None) == -1
    assert _ragged_call(L, lp, 6, 4, 16, 16) == -1
    assert _ragged_call(L, lp, 8, 4, 0, 16) == -1
    assert _ragged_call(L, lp, 8, 4, -3, 16) == -1


# ---- GPU ---------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("C,nc,nr,starts", [(1, 2500, 1000, 4), (1, 900, 1400, 2), (3, 1200, 800, 4)])
def test_lengths_at_the_strides_equal_the_equal_size_batch(cuda, C, nc, nr, starts):
    """A ragged batch runs register_step_kernel, one launch per iteration.  With every length at its stride it is bit for bit
    the equal-size batch in that form (GENPC_REGISTER_PERSIST=0), and within 1e-6 of the equal-size batch's default
    persistent form (partial sums in another order, as test_persistent_small_registration_equals_launch_per_iteration)."""
    import torch

    from genpc_b200 import _lib
    from genpc_b200.optim_registration.diff_obj_pose import RegistrationBatch

    pairs = make_pairs([(nc, nr)] * C, seed0=21)
    V = torch.from_numpy(np.stack([c for c, _ in pairs])).to(cuda)
    Rf = torch.from_numpy(np.stack([p for _, p in pairs])).to(cuda)
    iters = 40
    new = RegistrationBatch(V, Rf, n_starts=starts, lr=0.01, max_iters=iters,
                            complete_lengths=torch.full((C,), nc, dtype=torch.int32),
                            partial_lengths=torch.full((C,), nr, dtype=torch.int64, device=cuda))
    assert new.ragged
    new.run(iters)
    b = result(new)
    for persist in ("0", "1"):
        with _lib.tunable(GENPC_REGISTER_PERSIST=persist):
            old = RegistrationBatch(V, Rf, n_starts=starts, lr=0.01, max_iters=iters)
            assert not old.ragged
            if C > 1:   # the centre of a batch of C clouds is one reduction, a ragged batch's one per cloud: same start here
                old.center = new.center.clone()
            assert torch.equal(old.center, new.center)
            old.run(iters)
            a = result(old)
        if persist == "0":
            assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
        else:
            assert np.abs(a[0] - b[0]).max() <= 1e-6, np.abs(a[0] - b[0]).max()
            assert np.abs(a[1] - b[1]).max() <= 1e-6 * np.abs(a[1]).max()


def _solo(cuda, pair, starts, iters):
    import torch

    from genpc_b200.optim_registration.diff_obj_pose import RegistrationBatch

    c, p = pair
    rb = RegistrationBatch(torch.from_numpy(c[None]).to(cuda), torch.from_numpy(p[None]).to(cuda), n_starts=starts, lr=0.01,
                           max_iters=iters)
    rb.run(iters)
    return rb, result(rb)


@pytest.mark.gpu
def test_ragged_batch_vs_oracle_and_solo_runs(cuda):
    """Every start of every pair of the ragged batch over 60 iterations against its own RegistrationBatch (1e-6: the same
    arithmetic with the partial sums in another order); two ragged runs are bit-identical.  Every start of every pair over the
    first 12 iterations against OR.run on that pair alone at its own size (same float32 centre): losses within 1e-5, parameters
    of start 0 within 1e-5 and of the turned starts within 2e-4 -- Adam divides each gradient component by its own running
    magnitude, so rounding in a component near zero moves that parameter more than the loss (1.3e-4 measured on the 270 deg
    start of the first 2600 x 1400 pair on a B200, its solo run alike; test_dispatch_paths allows 1e-4).  (Over 60 iterations two
    2600 x 1400 pairs leave the oracle's trajectory by up to 3.9e-4 in the loss on a B200, and one by 4.9e-6 after 25; their
    solo runs, which the ragged run matches within 1e-6, do the same: the fp32 rounding of one step moves a neighbour choice
    and the trajectories part.)"""
    starts, iters = 4, 60
    pairs = make_pairs(RAGGED_SIZES)
    rb = ragged_batch(cuda, pairs, starts, iters)
    assert rb.Nc == 2600 and rb.Nr == 1400
    rb.run(iters)
    params, losses = result(rb)
    rb2 = ragged_batch(cuda, pairs, starts, iters)
    rb2.run(iters)
    assert all(np.array_equal(x, y) for x, y in zip((params, losses), result(rb2)))
    center = rb.center.cpu().numpy()
    for c, pair in enumerate(pairs):
        solo, (sp, sl) = _solo(cuda, pair, starts, iters)
        assert np.array_equal(solo.center.cpu().numpy()[0], center[c])
        mine = slice(c * starts, (c + 1) * starts)
        assert np.abs(params[mine] - sp).max() <= 1e-6, (c, np.abs(params[mine] - sp).max())
        assert (np.abs(losses[mine] - sl) <= 1e-6 * np.abs(sl)).all(), (c, np.abs(losses[mine] - sl).max())
    short = 12
    rb25 = ragged_batch(cuda, pairs, starts, short)
    rb25.run(short)
    p25, l25 = result(rb25)
    assert np.array_equal(l25, losses[:, :short])
    for c, pair in enumerate(pairs):
        for k in range(starts):   # the Ry(k * 90 deg) start of each scan
            eh, el = OR.run(pair[0], pair[1], short, lr=0.01, start=k, center=center[c])
            s = c * starts + k
            assert (np.abs(l25[s] - el) <= 1e-5 * np.abs(el)).all(), (c, k, np.abs(l25[s] - el).max())
            assert np.abs(p25[s] - eh[-1]).max() <= (1e-5 if k == 0 else 2e-4), (c, k, np.abs(p25[s] - eh[-1]).max())
    assert (losses[:, -1] < losses[:, 0]).all()


@pytest.mark.gpu
def test_padding_is_never_read(cuda):
    starts, iters = 4, 30
    pairs = make_pairs(RAGGED_SIZES)
    res = []
    for pad in (None, float("nan"), 1e30, -1e30):
        rb = ragged_batch(cuda, pairs, starts, iters, pad=pad)
        rb.run(iters)
        res.append(result(rb))
    for r in res[1:]:
        assert np.array_equal(r[0], res[0][0]) and np.array_equal(r[1], res[0][1])
    assert np.isfinite(res[0][1]).all()


@pytest.mark.gpu
def test_ragged_batches_launch_the_step_kernel_and_split_runs_equal_one_run(cuda):
    """110 pairs x 4 starts (the size of the Waymo object set) and a batch of 6 pairs small enough for the persistent kernel
    both launch register_step_kernel once per iteration, and nothing else.  Every pair of the 110 agrees with its solo run
    (persistent kernel) within 1e-6; run() split in calls equals one call bit for bit."""
    from test_dispatch_paths import launched_kernels

    starts, iters = 4, 12
    rng = np.random.default_rng(7)
    sizes = [(int(rng.integers(300, 2601)), int(rng.integers(300, 1401))) for _ in range(110)]
    pairs = make_pairs(sizes, seed0=1000)
    big = ragged_batch(cuda, pairs, starts, iters)
    _, ks = launched_kernels(lambda: big.run(iters))
    assert [k for k, _, _ in ks] == ["genpc::register_step_kernel<4>"] * iters, {k for k, _, _ in ks}
    bp, bl = result(big)
    for c, pair in enumerate(pairs):
        solo, (sp, sl) = _solo(cuda, pair, starts, iters)
        mine = slice(c * starts, (c + 1) * starts)
        assert np.abs(bp[mine] - sp).max() <= 1e-6, (c, np.abs(bp[mine] - sp).max())
        assert (np.abs(bl[mine] - sl) <= 1e-6 * np.abs(sl)).all(), (c, np.abs(bl[mine] - sl).max())
    small = pairs[:6]
    one = ragged_batch(cuda, small, starts, iters)
    _, ks = launched_kernels(lambda: one.run(iters))
    assert [k for k, _, _ in ks] == ["genpc::register_step_kernel<2>"] * iters, {k for k, _, _ in ks}
    two = ragged_batch(cuda, small, starts, iters)
    two.run(iters // 3)
    two.run(iters - iters // 3)
    assert all(np.array_equal(x, y) for x, y in zip(result(two), result(one)))


@pytest.mark.gpu
def test_large_ragged_batch_takes_the_step_kernel_and_matches_the_oracle(cuda):
    """Above the symmetric-path threshold an equal-size batch would take register_sym_scan_kernel; a ragged one launches
    only register_step_kernel (one per iteration: too many items to be co-resident).  Each pair matches its solo run within
    1e-6 and the oracle within 1e-5 on every loss; the parameters within 1e-4, as in test_dispatch_paths: Adam divides each
    gradient component by its own running magnitude, so rounding in a component near zero moves that parameter more than it
    moves the loss (4.2e-5 on a 6-D rotation entry of -0.024 after 4 steps of the 9500 x 8999 pair on a B200, solo run alike)."""
    from test_dispatch_paths import launched_kernels

    starts, iters = 2, 4
    pairs = make_pairs([(12000, 9000), (7001, 3333), (9500, 8999)], seed0=700)
    rb = ragged_batch(cuda, pairs, starts, iters)
    _, ks = launched_kernels(lambda: rb.run(iters))
    names = {k for k, _, _ in ks}
    assert names == {"genpc::register_step_kernel<4>"}, names
    assert sum(k == "genpc::register_step_kernel<4>" for k, _, _ in ks) == iters
    params, losses = result(rb)
    center = rb.center.cpu().numpy()
    for c, pair in enumerate(pairs):
        _, (sp, sl) = _solo(cuda, pair, starts, iters)
        mine = slice(c * starts, (c + 1) * starts)
        assert np.abs(params[mine] - sp).max() <= 1e-6, (c, np.abs(params[mine] - sp).max())
        assert (np.abs(losses[mine] - sl) <= 1e-6 * np.abs(sl)).all(), (c, np.abs(losses[mine] - sl).max())
        for k in range(starts):
            eh, el = OR.run(pair[0], pair[1], iters, lr=0.01, start=k, center=center[c])
            s = c * starts + k
            assert (np.abs(losses[s] - el) <= 1e-5 * np.abs(el)).all(), (c, k, np.abs(losses[s] - el).max())
            assert np.abs(params[s] - eh[-1]).max() <= 1e-4, (c, k, np.abs(params[s] - eh[-1]).max())


@pytest.mark.gpu
def test_object_pose_optimization_points_batch_equals_the_solo_calls(cuda):
    """The batched entry returns each pair's transform of the solo call.  The start each picks (argmin of the lowest loss) is
    compared first: a near tie flipped by rounding would otherwise show up as a large transform difference."""
    import torch

    from genpc_b200.optim_registration.diff_obj_pose import (RegistrationBatch, object_pose_optimization_points,
                                                             object_pose_optimization_points_batch)

    iters = 30
    pairs = make_pairs([(400, 300), (1500, 700), (800, 1200)], seed0=900)
    rb = ragged_batch(cuda, pairs, 4, iters + 1)
    rb.run(iters + 1)
    _, k_batch, lo_batch = rb.best()
    Ts = object_pose_optimization_points_batch([c for c, _ in pairs], [p for _, p in pairs], lr=0.01, iters=iters, device=cuda)
    assert Ts.shape == (3, 4, 4)
    for c, (comp, part) in enumerate(pairs):
        solo = RegistrationBatch(torch.from_numpy(comp[None]).to(cuda), torch.from_numpy(part[None]).to(cuda), n_starts=4,
                                 lr=0.01, max_iters=iters + 1)
        solo.run(iters + 1)
        _, k_solo, lo_solo = solo.best()
        assert int(k_batch[c]) == int(k_solo[0]), (c, rb.losses()[c * 4:(c + 1) * 4].min(1).values, solo.losses().min(1).values)
        assert abs(float(lo_batch[c]) - float(lo_solo[0])) <= 1e-6 * abs(float(lo_solo[0]))
        T = object_pose_optimization_points(comp, part, lr=0.01, iters=iters, device=cuda)
        assert np.abs(Ts[c] - T).max() <= 1e-5, (c, np.abs(Ts[c] - T).max())
