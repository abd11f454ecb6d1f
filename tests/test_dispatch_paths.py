"""The kernels the default dispatch picks at production sizes, against the oracle.

The host code chooses kernels by cloud size, batch size and SM count, so a test at a small size can miss the kernel a real
workload runs.  Every case here runs its call under torch.profiler, reads the launched kernels (and their grids) from the
exported trace and first asserts that the kernel it targets actually ran: a moved threshold fails the test instead of
quietly testing another kernel.  Thresholds are derived from the device's SM count.

- registration, symmetric path (S * Nc * Nr >= 2e8): register_sym_scan_kernel<2|4>, nn_prune_kernel + register_sims_kernel
  (pruned, from S = 20 at 16384^2), register_finish_kernel<256|512>: first-step loss and gradient and an 8-step trajectory
  against oracle/registration.py (1e-5 relative on losses, 1e-5 on the gradient scale and on the parameters);
- FPS above the cluster kernels' 144 points per thread and batches too large for the clusters: fps_gmem_kernel (the fusion
  step of reg_points at its real size, B > 1) and fps_reg_kernel<32, false>, bit for bit against oracle.fps, plus a float64
  check of the max-min rule that does not use the oracle;
- EMD with B close to or above the number of co-resident CTAs (group = 1: one cloud per CTA, or a CTA looping over clouds),
  bit for bit against the exhaustive scan and against oracle.emd_forward / oracle.emd_backward on sampled clouds;
- Chamfer with 512 to 1023 points in the cloud that sets the tile (two rows or queries per thread): nn_sym_kernel<2> for
  batches of at least 4 x SMs work items, nn_sym_gated_kernel<2> (host-fed forward and loss), nn_scan_kernel<2> (sharded
  partial scans and GENPC_CHAMFER_MODE=scan), bit for bit against the oracle."""
import json
import os
import tempfile
import time

import numpy as np
import pytest

import oracle
from oracle import registration as OR
from test_kernel_inventory import kernel_key
from util import lattice_cloud, shape_cloud

HERE = os.path.dirname(os.path.abspath(__file__))


def launched_kernels(fn):
    """fn() under torch.profiler (CUDA activity) -> (fn's result, [(kernel key, grid, duration in us)]) in launch order.
    The profiling window is padded by 20 ms on both sides of the call: traces of windows well under a millisecond were
    seen to come back without their kernels."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        time.sleep(0.02)
        out = fn()
        torch.cuda.synchronize()
        time.sleep(0.02)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    ks = [(kernel_key(e["name"]), tuple(e.get("args", {}).get("grid", ())), float(e.get("dur", 0.0)))
          for e in events if e.get("cat") == "kernel"]
    assert ks, "the profiler recorded no kernel launches"
    return out, ks


def grids(ks, key):
    """x-extent of the grid of every launch of kernel `key` (a key ending in '<': any instantiation); asserts that it ran."""
    g = [grid[0] for k, grid, _ in ks if (k.startswith(key) if key.endswith("<") else k == key)]
    assert g, f"{key} did not run; launched: {sorted({k for k, _, _ in ks})}"
    return g


def num_sms(dev):
    import torch

    return torch.cuda.get_device_properties(dev).multi_processor_count


# ---------------------------------------------------------------------------------------------------------------- registration
def make_pair(seed, nc, nr):
    from genpc_b200.synthetic import partial_view, rigid_perturb, superquadric

    comp = superquadric(seed, nc)
    part, _ = rigid_perturb(partial_view(comp, seed, nr), seed, max_rot_deg=20.0, max_t=0.05, scale_range=(0.7, 0.9))
    return comp, part


_PAIRS = {}


def pairs(C, nc, nr, seed0=100):
    key = (C, nc, nr, seed0)
    if key not in _PAIRS:
        _PAIRS[key] = [make_pair(seed0 + c, nc, nr) for c in range(C)]
    return _PAIRS[key]


def first_step_vs_oracle(cuda, C, n_starts, nc, nr, sample):
    """One Adam step of C * n_starts scans from perturbed starting poses; loss and gradient (adam_m / (1 - beta1)) of the
    sampled scans against OR.loss_and_grad.  -> the kernels launched."""
    import torch

    from genpc_b200.optim_registration.diff_obj_pose import RegistrationBatch

    pr = pairs(C, nc, nr)
    comp = torch.from_numpy(np.stack([p[0] for p in pr])).to(cuda)
    part = torch.from_numpy(np.stack([p[1] for p in pr])).to(cuda)
    rb = RegistrationBatch(comp, part, n_starts=n_starts, lr=0.01)
    g = torch.Generator().manual_seed(C * n_starts)
    rb.params += (torch.randn(rb.params.shape, generator=g) * 0.02).to(cuda)
    p0 = rb.params.cpu().numpy().copy()
    _, ks = launched_kernels(lambda: rb.run(1))
    m = rb.adam_m.cpu().numpy()
    loss = rb.losses().cpu().numpy()[:, 0]
    center = rb.center.cpu().numpy()
    for s in sample:
        c = s // n_starts
        eloss, egrad, _ = OR.loss_and_grad(p0[s], pr[c][0], center[c], pr[c][1])
        assert abs(loss[s] - eloss) <= 1e-5 * abs(eloss), (s, loss[s], eloss)
        got = m[s] / np.float32(1.0 - 0.9)
        assert np.abs(got - egrad).max() <= 1e-5 * np.abs(egrad).max() + 1e-7, (s, got, egrad)
    assert np.isfinite(loss).all() and np.isfinite(m).all()
    return ks


def sample_scans(S, extra=()):
    return sorted({0, S // 2, S - 1, *[e for e in extra if 0 <= e < S]})


@pytest.mark.gpu
def test_registration_c3_pruned_sym_finish512_vs_oracle(cuda):
    """BASELINE C3: 64 scans x 16384^2, one start -> pruned scan + symmetric scan + register_finish_kernel<512>."""
    S = 64
    ks = first_step_vs_oracle(cuda, S, 1, 16384, 16384, sample_scans(S, (1, 13, 27, 45, 50)))
    grids(ks, "genpc::nn_prune_kernel<")
    grids(ks, "genpc::register_sims_kernel")
    grids(ks, "genpc::register_sym_scan_kernel<4>")
    assert grids(ks, "genpc::register_finish_kernel<512>") == [S * 16384 // 512]


@pytest.mark.gpu
def test_registration_multistart_pruned_sym_vs_oracle(cuda):
    """16 clouds x 4 starts at 16384^2: the pruned scan's per-start indexing (qdiv / tdiv) and the finish kernel's cloud of a scan."""
    S = 64
    ks = first_step_vs_oracle(cuda, 16, 4, 16384, 16384, sample_scans(S, (1, 2, 3, 22, 41, 61)))
    grids(ks, "genpc::nn_prune_kernel<")
    grids(ks, "genpc::register_sym_scan_kernel<4>")
    grids(ks, "genpc::register_finish_kernel<512>")


@pytest.mark.gpu
def test_registration_8_scans_exhaustive_sym_finish256_vs_oracle(cuda):
    """The 8-GPU bench line's share per rank: 8 scans x 16384^2 -> exhaustive symmetric scan + register_finish_kernel<256>."""
    S = 8
    ks = first_step_vs_oracle(cuda, S, 1, 16384, 16384, range(S))
    assert not any(k.startswith("genpc::nn_prune_kernel") for k, _, _ in ks)
    grids(ks, "genpc::register_sym_scan_kernel<4>")
    assert grids(ks, "genpc::register_finish_kernel<256>") == [S * 16384 // 256]


@pytest.mark.gpu
def test_registration_sym_scan_two_rows_per_thread_vs_oracle(cuda):
    """512 <= Nr < 1024 on the symmetric path: register_sym_scan_kernel<2> (8 scans, 30000 x 900)."""
    ks = first_step_vs_oracle(cuda, 4, 2, 30000, 900, range(8))
    grids(ks, "genpc::register_sym_scan_kernel<2>")
    grids(ks, "genpc::register_finish_kernel<512>")


@pytest.mark.gpu
def test_registration_pruned_clouds_above_16384_points_vs_oracle(cuda):
    """24 scans x 20000^2: more than 256 blocks of 64 points per cloud -> nn_prune_kernel<16>."""
    ks = first_step_vs_oracle(cuda, 24, 1, 20000, 20000, sample_scans(24, (5,)))
    grids(ks, "genpc::nn_prune_kernel<16>")
    grids(ks, "genpc::register_finish_kernel<512>")


@pytest.mark.gpu
def test_registration_single_cloud_four_starts_finish128_vs_oracle(cuda):
    """1 cloud x 4 starts at 16384^2: symmetric path, exhaustive (too few query groups for the pruned scan), the finish
    kernel's smallest form register_finish_kernel<128>."""
    ks = first_step_vs_oracle(cuda, 1, 4, 16384, 16384, range(4))
    assert not any(k.startswith("genpc::nn_prune_kernel") for k, _, _ in ks)
    grids(ks, "genpc::register_finish_kernel<128>")


@pytest.mark.gpu
@pytest.mark.parametrize("shape,iters,key", [
    ((4, 4, 8000, 900), 1, "genpc::register_step_kernel<2>"),
    ((5, 4, 3000, 3000), 1, "genpc::register_step_kernel<4>"),
    ("sms/4, 2, 1024, 900", 8, "genpc::register_persistent_kernel<2,1024>"),
    ("sms/8, 1, 2048, 2048", 8, "genpc::register_persistent_kernel<4,1024>"),
    ((1, 4, 1200, 800), 8, "genpc::register_persistent_kernel<1,256>")])
def test_registration_small_problem_kernels_vs_oracle(cuda, shape, iters, key):
    """Below S * Nc * Nr = 2e8 one launch runs an iteration (run(1)) or all of them (cooperative, persistent); its queries per
    thread and target span follow the problem size, and the persistent kernel needs its grid co-resident (sized here from
    the SM count: 2 work items per SM).  The first and last scan against OR.run (multi-start k begins at Ry(k * 90 deg)):
    every loss within 1e-5 relative, the final parameters within 1e-4.  (Adam divides each gradient component by its own
    running magnitude, so rounding differences in a component near zero move that parameter by more than they move the
    loss: 2.1e-5 after 8 steps was measured on the start at 270 deg of the 1200 x 800 pair on a B200.)"""
    import torch

    from genpc_b200.optim_registration.diff_obj_pose import RegistrationBatch

    if isinstance(shape, str):
        div, starts, nc, nr = (int(v.strip("sms/")) for v in shape.split(","))
        C = (2 * num_sms(cuda) // div + starts - 1) // starts
    else:
        C, starts, nc, nr = shape
    pr = pairs(C, nc, nr, seed0=300)
    comp = torch.from_numpy(np.stack([p[0] for p in pr])).to(cuda)
    part = torch.from_numpy(np.stack([p[1] for p in pr])).to(cuda)
    rb = RegistrationBatch(comp, part, n_starts=starts, lr=0.01, max_iters=iters)
    _, ks = launched_kernels(lambda: rb.run(iters))
    grids(ks, key)
    losses, params, center = rb.losses().cpu().numpy(), rb.params.cpu().numpy(), rb.center.cpu().numpy()
    for s in (0, rb.S - 1):
        c, k = divmod(s, starts)
        eh, el = OR.run(pr[c][0], pr[c][1], iters, lr=0.01, start=k, center=center[c])
        assert (np.abs(losses[s] - el) <= 1e-5 * np.abs(el)).all(), (s, np.abs(losses[s] - el).max())
        assert np.abs(params[s] - eh[-1]).max() <= 1e-4, (s, np.abs(params[s] - eh[-1]).max())


@pytest.mark.gpu
def test_registration_c3_trajectory_vs_oracle(cuda):
    """8 Adam iterations of the C3 batch (pruned + finish<512>); scans 0 and 63 against OR.run at every step."""
    import torch

    from genpc_b200.optim_registration.diff_obj_pose import RegistrationBatch

    S, iters = 64, 8
    pr = pairs(S, 16384, 16384)
    comp = torch.from_numpy(np.stack([p[0] for p in pr])).to(cuda)
    part = torch.from_numpy(np.stack([p[1] for p in pr])).to(cuda)
    rb = RegistrationBatch(comp, part, n_starts=1, lr=0.01, max_iters=iters)
    hist = [rb.params.cpu().numpy().copy()]

    def step():
        rb.run(1)
        return rb.params.cpu().numpy().copy()

    p1, ks = launched_kernels(step)
    grids(ks, "genpc::nn_prune_kernel<")
    grids(ks, "genpc::register_finish_kernel<512>")
    hist.append(p1)
    for _ in range(iters - 1):
        hist.append(step())
    hist = np.stack(hist)
    losses = rb.losses().cpu().numpy()
    for s in (0, S - 1):
        eh, el = OR.run(pr[s][0], pr[s][1], iters, lr=0.01, center=rb.center[s].cpu().numpy())
        assert (np.abs(losses[s] - el) <= 1e-5 * np.abs(el)).all(), (s, np.abs(losses[s] - el).max())
        assert np.abs(hist[:, s] - eh).max() <= 1e-5, (s, np.abs(hist[:, s] - eh).max())


# ------------------------------------------------------------------------------------------------------------------------- FPS
def fps_vs_oracle(cuda, a, K, start, key):
    import torch

    from genpc_b200.fps import furthest_point_sample

    x = torch.from_numpy(a).to(cuda)
    (idx, seq), ks = launched_kernels(lambda: furthest_point_sample(x, K, start, return_seq=True))
    g = grids(ks, key)
    eidx, eseq = oracle.fps(a, K, start, True)
    idx, seq = idx.cpu().numpy(), seq.cpu().numpy()
    assert np.array_equal(idx, eidx), f"{(idx != eidx).sum()} indices differ, first at {np.argwhere(idx != eidx)[0]}"
    assert np.array_equal(seq.view(np.int32), eseq.view(np.int32))
    return idx, seq, g, ks


def fusion_cloud(cuda):
    """reg_points' fusion input at its real size: the committed C1 scan (71 372 points) followed by the 163 840 surface
    samples of a generated mesh (ScaleAdapter's glb sample count) -> [235 212, 3] float32."""
    import torch

    from genpc_b200.synthetic import superquadric_mesh
    from genpc_b200.utils.glb import sample_mesh

    scan = np.load(os.path.join(HERE, "golden", "scan_01184_xyz.npz"))["xyz"].astype(np.float32)
    v, f, _ = superquadric_mesh(3)
    # the scan spans about a metre: place the mesh samples over it as the registered glb cloud would be
    lo, hi = scan.min(0), scan.max(0)
    v = v * np.float32((hi - lo).max()) + ((lo + hi) / 2).astype(np.float32)
    xyz, _ = sample_mesh(torch.from_numpy(v).to(cuda), torch.from_numpy(f).to(cuda), 163840, seed=5)
    return np.ascontiguousarray(np.concatenate([scan, xyz.cpu().numpy()])[None], np.float32)


@pytest.mark.gpu
def test_fps_fusion_size_gmem_kernel_vs_oracle_and_float64(cuda):
    """235 212 -> 20 000 (reg_xyz.py's n_fused): one CTA, running distances in global memory.  Besides the oracle: every
    one of the first 200 picks is the float64 max-min distance to the picks before it (within 2^-20), attained by idx[s]."""
    a = fusion_cloud(cuda)
    assert a.shape == (1, 71372 + 163840, 3)
    idx, seq, g, ks = fps_vs_oracle(cuda, a, 20000, 0, "genpc::fps_gmem_kernel")
    assert g == [1]
    ms = sum(d for k, _, d in ks if k == "genpc::fps_gmem_kernel") / 1e3
    print(f"fps_gmem_kernel 235212 -> 20000: {ms:.1f} ms")
    p = a[0].astype(np.float64)
    run = np.full(p.shape[0], np.inf)
    assert idx[0, 0] == 0 and np.isinf(seq[0, 0])
    for s in range(1, 200):
        run = np.minimum(run, ((p - p[idx[0, s - 1]]) ** 2).sum(1))
        best = run.max()
        assert abs(float(seq[0, s]) - best) <= 2.0 ** -20 * best, (s, seq[0, s], best)
        assert run[idx[0, s]] >= best * (1 - 2.0 ** -20), (s, idx[0, s], run[idx[0, s]], best)


@pytest.mark.gpu
@pytest.mark.parametrize("N,key", [(147456, "genpc::fps_cluster_kernel<"), (147457, "genpc::fps_gmem_kernel"),
                                   (60000, "genpc::fps_cluster_kernel<4,16,false>")])
def test_fps_both_sides_of_the_cluster_limit(cuda, N, key):
    """144 points per thread is the cluster kernels' limit: 147 456 points run 16-CTA clusters, one more point the gmem kernel.
    (60 000 points: the 16-CTA form with 4 points per thread, which 48 < points per thread <= 64 selects.)"""
    a = shape_cloud(N, 1, N)
    fps_vs_oracle(cuda, a, 300, 7, key)


@pytest.mark.gpu
@pytest.mark.parametrize("N,key", [(32769, "genpc::fps_gmem_kernel"), (40000, "genpc::fps_gmem_kernel"),
                                   (16385, "genpc::fps_reg_kernel<32,false>"), (20000, "genpc::fps_reg_kernel<32,false>"),
                                   (32768, "genpc::fps_reg_kernel<32,false>")])
def test_fps_batches_beyond_the_clusters(cuda, N, key):
    """B = SMs / 8 + 1 clouds cannot all get an 8-CTA cluster: one CTA per cloud, the registers-only kernel up to 32 points
    per thread and the gmem kernel above (its per-cloud workspace offset with B > 1); start = N - 1."""
    B = num_sms(cuda) // 8 + 1
    a = shape_cloud(N + 3, B, N)
    _, _, g, _ = fps_vs_oracle(cuda, a, 256, N - 1, key)
    assert g == [B]


@pytest.mark.gpu
def test_fps_lattice_ties_above_the_cluster_limit(cuda):
    """150 000 integer-lattice points (exact distance ties everywhere): the gmem kernel's lowest-index tie rule."""
    a = lattice_cloud(9, 1, 150000, side=40)
    fps_vs_oracle(cuda, a, 300, 0, "genpc::fps_gmem_kernel")


# ------------------------------------------------------------------------------------------------------------------------- EMD
EMD_EPS, EMD_ITERS = 0.005, 50


def emd_run(cuda, x1, x2, knob=None):
    import torch

    from genpc_b200 import _lib
    from genpc_b200.loss_functions import emdModule

    t1, t2 = torch.from_numpy(x1).to(cuda), torch.from_numpy(x2).to(cuda)
    with _lib.tunable(GENPC_EMD_PRUNE=knob):
        (d, a), ks = launched_kernels(lambda: emdModule()(t1, t2, EMD_EPS, EMD_ITERS))
    return d.cpu().numpy(), a.cpu().numpy(), ks


def emd_inputs(B, n, seed):
    rng = np.random.default_rng(seed)
    return rng.random((B, n, 3), dtype=np.float32), rng.random((B, n, 3), dtype=np.float32)


def emd_vs_oracle(x1, x2, d, a, clouds):
    for b in clouds:
        ed, ea = oracle.emd_forward(x1[b:b + 1], x2[b:b + 1], EMD_EPS, EMD_ITERS)
        assert np.array_equal(a[b], ea[0]), f"cloud {b}: {(a[b] != ea[0]).sum()} assignments differ"
        assert np.array_equal(d[b].view(np.int32), ed[0].view(np.int32)), f"cloud {b}"
    assert (a >= 0).all()


@pytest.mark.gpu
def test_emd_batch_512_more_clouds_than_ctas(cuda):
    """B = 512 (the largest batch accepted), n = 1024: the pruned kernel (3 CTAs per SM) runs fewer CTAs than clouds, so CTAs
    loop over several clouds.  Bit for bit equal to the exhaustive scan (one cloud per CTA at this B), sampled clouds (among
    them the first and last of a CTA's first and second round) against the oracle, and the backward against the oracle."""
    import torch

    from genpc_b200 import emd as E

    B, n = 512, 1024
    x1, x2 = emd_inputs(B, n, 512)
    d, a, ks = emd_run(cuda, x1, x2)
    (grid,) = grids(ks, "genpc::emd_auction_kernel<4,3>")
    assert grid < B, grid
    d0, a0, ks0 = emd_run(cuda, x1, x2, "0")
    assert grids(ks0, "genpc::emd_auction_kernel<0,5>") == [B]
    assert np.array_equal(a, a0), f"{(a != a0).sum()} assignments differ"
    assert np.array_equal(d.view(np.int32), d0.view(np.int32))
    emd_vs_oracle(x1, x2, d, a, sorted({0, 1, grid - 1, grid, min(2 * grid - 1, B - 1), 300, B - 2, B - 1}))
    # backward: gradxyz = 2 * graddist * (xyz1 - xyz2[assignment]), elementwise
    gd = np.random.default_rng(1).random((B, n), dtype=np.float32)
    t1, t2 = torch.from_numpy(x1).to(cuda), torch.from_numpy(x2).to(cuda)
    gx = torch.zeros(B, n, 3, device=cuda)
    _, kb = launched_kernels(lambda: E.backward(t1, t2, gx, torch.from_numpy(gd).to(cuda), torch.from_numpy(a).to(cuda)))
    assert grids(kb, "genpc::emd_grad_kernel") == [B * n // 256]
    eg = oracle.emd_backward(x1, x2, gd, a)
    assert np.array_equal(gx.cpu().numpy().view(np.int32), eg.view(np.int32))


@pytest.mark.gpu
@pytest.mark.parametrize("B,knob,key", [(300, None, "genpc::emd_auction_kernel<4,3>"), (400, "0", "genpc::emd_auction_kernel<0,5>")])
def test_emd_batch_one_cloud_per_cta(cuda, B, knob, key):
    """resident / 2 < B < resident: group = 1, one cloud per CTA (the pruned kernel's default at B = 300, the exhaustive one
    at B = 400); sampled clouds against the oracle."""
    n = 1024
    x1, x2 = emd_inputs(B, n, B)
    d, a, ks = emd_run(cuda, x1, x2, knob)
    assert grids(ks, key) == [B]
    emd_vs_oracle(x1, x2, d, a, sorted({0, 1, B // 3, B // 2, B - 2, B - 1}))


# ------------------------------------------------------------------------------------------------------------------------- kNN
@pytest.mark.gpu
@pytest.mark.parametrize("k", range(1, 33))
def test_knn_mean_distance_every_list_size(cuda, k):
    """genpc_knn_mean_distance instantiates one kernel per k (1..32, the mean runs over the whole list): every one of them
    against the oracle, bit for bit, on a lattice cloud (exact ties) and a shape cloud, with and without the point itself."""
    import torch

    from genpc_b200.reg_xyz import knn_mean_distance

    xs = (lattice_cloud(k, 1, 1500, side=8)[0], shape_cloud(k + 40, 1, 1500)[0])
    ts = [torch.from_numpy(x).to(cuda) for x in xs]
    got, ks = launched_kernels(lambda: [knn_mean_distance(t, k, inc).cpu().numpy() for t in ts for inc in (True, False)])
    assert grids(ks, f"genpc::knn_mean_kernel<{k}>")
    exp = [oracle.knn_mean_distance(x, k, inc) for x in xs for inc in (True, False)]
    for g, e in zip(got, exp):
        assert np.array_equal(g.view(np.int32), e.view(np.int32))


# ------------------------------------------------------------------------------------- Chamfer, two rows / queries per thread
def chamfer_batch(seed, B, n):
    """B clouds of n points: shape clouds, every third one an integer-lattice cloud (exact distance ties)."""
    x = shape_cloud(seed, B, n)
    x[::3] = lattice_cloud(seed + 1, B, n, side=8)[::3]
    return x


def same_as_oracle(got, exp, tag):
    for g, e, name in zip(got, exp, ("dist1", "dist2", "idx1", "idx2")):
        bad = g.view(np.int32) != e.view(np.int32)
        assert not bad.any(), f"{tag} {name}: {bad.sum()} of {g.size} differ, first at {np.argwhere(bad)[0]}"


@pytest.mark.gpu
@pytest.mark.parametrize("per_sm,extra,N,M", [(2, 8, 1000, 777), (4, 4, 300, 512)])
def test_chamfer_sym_kernel_two_rows_per_thread_vs_oracle(cuda, per_sm, extra, N, M):
    """B = per_sm * SMs + extra clouds whose larger side has 512 to 1023 points: two rows per thread, and at least 4 x SMs work
    items, so one CTA per item (nn_sym_kernel<2>, not the balanced form).  1000 x 777: two row tiles per cloud; 300 x 512:
    the smallest clouds the symmetric path takes, one row tile, the second cloud as rows."""
    import torch

    from genpc_b200.loss_functions import chamfer_3DDist

    B = per_sm * num_sms(cuda) + extra
    a, b = chamfer_batch(N, B, N), chamfer_batch(M + 1, B, M)
    ta, tb = torch.from_numpy(a).to(cuda), torch.from_numpy(b).to(cuda)
    got, ks = launched_kernels(lambda: [t.cpu().numpy() for t in chamfer_3DDist()(ta, tb)])
    grids(ks, "genpc::nn_sym_kernel<2>")
    same_as_oracle(got, oracle.chamfer_forward(a, b), f"{B} x {N} x {M}")


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,M,chunks", [(64, 1000, 600, 4), (5, 513, 1023, 2)])
def test_host_fed_forward_two_rows_per_thread_vs_oracle(cuda, B, N, M, chunks):
    """forward_from_host with fewer than 1024 points in the larger cloud: nn_sym_gated_kernel<2>, from pinned and from pageable
    host memory."""
    import torch

    from genpc_b200.loss_functions import chamfer_3DDist

    a, b = chamfer_batch(B + N, B, N), chamfer_batch(B + M + 1, B, M)
    exp = oracle.chamfer_forward(a, b)
    for pin in (True, False):
        ha, hb = torch.from_numpy(a), torch.from_numpy(b)
        if pin:
            ha, hb = ha.pin_memory(), hb.pin_memory()
        got, ks = launched_kernels(
            lambda: [t.detach().cpu().numpy() for t in chamfer_3DDist().forward_from_host(ha, hb, device=cuda, chunks=chunks)[:4]])
        grids(ks, "genpc::nn_sym_gated_kernel<2>")
        same_as_oracle(got, exp, f"{B} x {N} x {M}, pinned={pin}")


@pytest.mark.gpu
def test_loss_from_host_two_rows_per_thread_equals_device_call(cuda):
    """get_loss_from_host('cd_l2') through nn_sym_gated_kernel<2> gives the loss of the device-resident call."""
    import torch

    from genpc_b200.utils.loss_util import Completionloss

    a, b = chamfer_batch(70, 64, 1000), chamfer_batch(71, 64, 600)
    crit = Completionloss("cd_l2")
    ref = float(crit.get_loss(torch.from_numpy(a).to(cuda), torch.from_numpy(b).to(cuda)))
    (loss, _, _), ks = launched_kernels(
        lambda: crit.get_loss_from_host(torch.from_numpy(a).pin_memory(), torch.from_numpy(b).pin_memory(), device=cuda, chunks=4))
    grids(ks, "genpc::nn_sym_gated_kernel<2>")
    assert float(loss) == ref


@pytest.mark.gpu
@pytest.mark.parametrize("nq", [512, 1023])
def test_partial_scan_two_queries_per_thread_merges_to_the_oracle(cuda, nq):
    """genpc_nn_partial_packed with 512 and 1023 queries (the edges of two queries per thread, nn_scan_kernel<2>) against three
    ragged shards of a 30 011-point lattice cloud, global indices from idx_base: the min-merge of the packed words is
    oracle.nn_distance against the whole cloud, distance bits and lowest indices.  Queries sit at lattice and half-integer
    positions (several equidistant targets, often in different shards)."""
    import torch

    from genpc_b200.sharded import nn_partial_packed, nn_unpack

    t = lattice_cloud(80, 1, 30011, side=40)
    rng = np.random.default_rng(nq)
    q = (rng.integers(0, 40, (1, nq, 3)) + 0.5 * rng.integers(0, 2, (1, nq, 3))).astype(np.float32)
    tq, tt = torch.from_numpy(q).to(cuda), torch.from_numpy(t).to(cuda)
    cuts = (0, 7001, 19999, 30011)

    def scan():
        parts = [nn_partial_packed(tq, tt[:, lo:hi], lo) for lo, hi in zip(cuts[:-1], cuts[1:])]
        d, i = nn_unpack(torch.stack(parts).min(0).values)
        return d.cpu().numpy(), i.cpu().numpy()

    (d, i), ks = launched_kernels(scan)
    assert len(grids(ks, "genpc::nn_scan_kernel<2>")) == 3
    ed, ei = oracle.nn_distance(q, t)
    assert np.array_equal(d.view(np.int32), ed.view(np.int32)), f"{(d != ed).sum()} distances differ"
    assert np.array_equal(i, ei), f"{(i != ei).sum()} indices differ"


@pytest.mark.gpu
def test_scan_mode_two_queries_per_thread_vs_oracle(cuda):
    """GENPC_CHAMFER_MODE=scan (one scan per direction) with 700 points in the smaller cloud: nn_scan_kernel<2>."""
    import torch

    from genpc_b200 import _lib
    from genpc_b200.loss_functions import chamfer_3DDist

    a, b = chamfer_batch(90, 4, 2600), chamfer_batch(91, 4, 700)
    ta, tb = torch.from_numpy(a).to(cuda), torch.from_numpy(b).to(cuda)
    with _lib.tunable(GENPC_CHAMFER_MODE="scan"):
        got, ks = launched_kernels(lambda: [t.cpu().numpy() for t in chamfer_3DDist()(ta, tb)])
    grids(ks, "genpc::nn_scan_kernel<2>")
    same_as_oracle(got, oracle.chamfer_forward(a, b), "scan mode, 4 x 2600 x 700")


# ------------------------------------------------------------------------------------------------------------ Chamfer backward
@pytest.mark.gpu
def test_fused_loss_backward_with_unaligned_gradient_arrays(cuda):
    """genpc_chamfer_loss_backward (the fused loss step's gradient) into gradient arrays that are only 4-byte aligned: the
    scalar form chamfer_grad_kernel<false, true>, against the oracle's double-accumulated backward (cd_l2 weights)."""
    import torch

    from genpc_b200 import _lib

    B, N, M = 2, 1500, 4100
    a, b = shape_cloud(80, B, N), shape_cloud(81, B, M)
    d1, d2, i1, i2 = oracle.chamfer_forward(a, b)
    ta, tb = torch.from_numpy(a).to(cuda), torch.from_numpy(b).to(cuda)
    td = [torch.from_numpy(x).to(cuda) for x in (d1, d2, i1, i2)]
    up = torch.ones((), device=cuda)

    def off(n):
        flat = torch.zeros(n + 5, device=cuda)
        v = flat[1:1 + n]
        assert v.data_ptr() % 8 != 0
        return v

    ga, gb = off(B * N * 3).view(B, N, 3), off(B * M * 3).view(B, M, 3)

    def call():
        rc = _lib.lib().genpc_chamfer_loss_backward(_lib.ptr(ta), _lib.ptr(tb), _lib.ptr(td[0]), _lib.ptr(td[1]),
                                                    _lib.ptr(td[2]), _lib.ptr(td[3]), _lib.ptr(up), 0, 1.0, 1.0,
                                                    _lib.ptr(ga), _lib.ptr(gb), B, N, M, _lib.current_stream(cuda))
        _lib.check(rc, "genpc_chamfer_loss_backward")

    _, ks = launched_kernels(call)
    grids(ks, "genpc::chamfer_grad_kernel<false,true>")
    e1, e2 = oracle.chamfer_backward(a, b, np.full((B, N), 1.0 / (B * N), np.float32), np.full((B, M), 1.0 / (B * M), np.float32),
                                     i1, i2)
    assert np.abs(ga.cpu().numpy() - e1).max() <= 1e-5 * np.abs(e1).max()
    assert np.abs(gb.cpu().numpy() - e2).max() <= 1e-5 * np.abs(e2).max()
