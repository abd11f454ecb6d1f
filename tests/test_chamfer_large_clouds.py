"""The two-level pruned scan (csrc/nn_grid.cuh) at the target sizes where nn_prune2_kernel<SBR> changes form, against three
references: the exhaustive kernels (GENPC_CHAMFER_PRUNE=0, all four outputs bit for bit), the CPU oracle on sampled queries
(distance bits and lowest index), and, for BASELINE C5, a float64 KD-tree check of every query that shares no code with the
kernels.

launch_prune2 keeps a lane's superblock distances in SBR registers, SBR = 1 / 2 / 4 / 8 / 16 for up to 32 / 64 / 128 / 256 /
512 superblocks of 4096 points.  A superblock id lives in the 9 low bits of the selection key, so GR_MAX_N = 2 097 152 points
is the largest target cloud the path takes.  Target sizes one point past a boundary leave a last superblock of one point.
To keep the exhaustive reference cheap, most pairs are asymmetric: about 50 000 queries drawn from the other scene cloud
against the target size under test, so the query -> target direction runs the SBR under test.

Every case first asserts from the profiler trace that the instantiation it targets ran (or, past the path's limits, that no
nn_prune2_kernel ran): a moved threshold fails the test instead of quietly testing another kernel."""
import time

import numpy as np
import pytest

import oracle
from test_chamfer_prune import run, same
from test_dispatch_paths import launched_kernels
from util import lattice_cloud

pytestmark = pytest.mark.gpu

P2 = "genpc::nn_prune2_kernel<"
QUERIES = 50000
SAMPLES = 2048          # oracle queries per direction
GR_MAX_N = 2 * 1024 * 1024


@pytest.fixture(scope="module")
def scene():
    """One LiDAR-like scene pair (the C5 generator) of GR_MAX_N + 1 points: targets are prefixes of the first cloud, queries
    prefixes of the second (its perturbed twin)."""
    from genpc_b200.synthetic import lidar_scene_pair

    a, b = lidar_scene_pair(GR_MAX_N + 1, 0)
    return a.numpy(), b.numpy()


def traced(a, b, dev, prune):
    """run() under the profiler -> (outputs, prune counters, {kernel key: [grid of every launch]})."""
    (out, st), ks = launched_kernels(lambda: run(a, b, dev, prune))
    launched = {}
    for k, grid, _ in ks:
        launched.setdefault(k, []).append(grid)
    return out, st, launched


def ran(launched, key):
    assert key in launched, f"{key} did not run; launched: {sorted(launched)}"
    return launched[key]


def no_grid_scan(launched):
    assert not any(k.startswith(P2) for k in launched), sorted(k for k in launched if k.startswith(P2))


def oracle_samples(a, b, got, seed):
    """Sampled queries of both directions of chamfer(a, b) (SAMPLES per direction, spread over the clouds, the first and last
    query of each cloud included) against the whole other cloud: distance bits and index equal.  -> seconds spent."""
    t0 = time.perf_counter()
    rng = np.random.default_rng(seed)
    B = a.shape[0]
    for q, t, d, i, name in ((a, b, got[0], got[2], "dist1/idx1"), (b, a, got[1], got[3], "dist2/idx2")):
        n = q.shape[1]
        for c in range(B):
            s = np.unique(np.concatenate([[0, n - 1], rng.choice(n, min(n, -(-SAMPLES // B)), replace=False)]))
            ed, ei = oracle.nn_distance(q[c:c + 1, s], t[c:c + 1])
            bad = (d[c, s].view(np.int32) != ed[0].view(np.int32)) | (i[c, s] != ei[0])
            assert not bad.any(), f"{name}, cloud {c}: {bad.sum()} of {s.size} sampled queries differ, first query {s[bad][0]}"
    return time.perf_counter() - t0


def float64_check(q, t, d, i):
    """Every query of one direction against a float64 KD-tree of the targets (scipy, not the oracle): with e the float64 squared
    distance to the returned target and m < m2 the two smallest, d is e to float32 accuracy, e is the minimum to within the
    rounding of the float32 distances, and the index is the nearest one wherever the nearest is not nearly tied."""
    from scipy.spatial import cKDTree

    q64, t64 = q.astype(np.float64), t.astype(np.float64)
    assert i.min() >= 0 and i.max() < t.shape[0]
    r, j = cKDTree(t64).query(q64, k=2, workers=-1)
    m, m2 = r[:, 0] ** 2, r[:, 1] ** 2
    e = ((q64 - t64[i]) ** 2).sum(1)
    bad = np.abs(d.astype(np.float64) - e) > 1e-6 * e
    assert not bad.any(), f"{bad.sum()} distances are not the float64 distance to their index, first query {np.argmax(bad)}"
    bad = e > m * (1 + 2e-6)
    assert not bad.any(), f"{bad.sum()} indices are not a nearest target, first query {np.argmax(bad)}"
    bad = (m2 > m * (1 + 1e-5)) & (i != j[:, 0])
    assert not bad.any(), f"{bad.sum()} indices differ from a clearly nearest target, first query {np.argmax(bad)}"


def superblocks(n):
    return -(-(-(-n // 64)) // 64)


# ------------------------------------------------------------------------------------------------------------ SBR boundaries
@pytest.mark.parametrize("nt,sbr", [(524288, 4), (524289, 8), (1048576, 8), (1048577, 16), (1500001, 16), (GR_MAX_N, 16)])
def test_grid_scan_superblock_register_edges(cuda, scene, nt, sbr):
    """50 000 queries x nt scene targets on both sides of each SBR boundary and at GR_MAX_N (superblock id 511): the default
    path (sampled probe, then the scan) and GENPC_CHAMFER_PRUNE=2 (no probe), both bit-identical to the exhaustive kernels."""
    assert 32 * sbr >= superblocks(nt) > 16 * sbr
    a, b = scene
    q, t = b[None, :QUERIES], a[None, :nt]
    ref, st0 = run(q, t, cuda, "0")
    assert st0[2] == 0
    for prune in (False, "2"):
        got, st, launched = traced(q, t, cuda, prune)
        ran(launched, f"{P2}{sbr},false>")
        assert (f"{P2}{sbr},true>" in launched) == (prune is False), sorted(launched)   # the probe runs unless forced
        assert st[2] > 0, st                                                            # the pruned scan did the work
        same(got, ref, f"{nt} targets, prune={prune} vs exhaustive")
    secs = oracle_samples(q, t, got, nt)
    print(f"{QUERIES} x {nt}: oracle samples {secs:.2f} s")


# ----------------------------------------------------------------------------------------------------------------------- C5
def test_c5_full_size_default_path(cuda):
    """BASELINE C5 as the README times it: chamfer_3DDist() on lidar_scene_pair(1 000 000, 0), no knob -> 245 superblocks per
    cloud, nn_prune2_kernel<8> with its probe in both directions.  Bit-identical to the exhaustive kernels, sampled queries
    against the oracle, and every query of both directions against a float64 KD-tree."""
    from genpc_b200.synthetic import lidar_scene_pair

    a, b = (x.numpy()[None] for x in lidar_scene_pair(1_000_000, 0))
    got, st, launched = traced(a, b, cuda, False)
    ran(launched, f"{P2}8,true>")
    ran(launched, f"{P2}8,false>")
    assert st[2] > 0, st
    ref, _ = run(a, b, cuda, "0")
    same(got, ref, "C5 vs exhaustive")
    secs = oracle_samples(a, b, got, 5)
    t0 = time.perf_counter()
    float64_check(a[0], b[0], got[0][0], got[2][0])
    float64_check(b[0], a[0], got[1][0], got[3][0])
    print(f"C5: oracle samples {secs:.2f} s, KD-tree check {time.perf_counter() - t0:.2f} s")


# --------------------------------------------------------------------------------------------------------------------- ties
@pytest.mark.parametrize("targets", ["lattice", "every_point_twice"])
def test_grid_scan_ties_at_16_superblock_registers(cuda, targets):
    """1.2M integer-lattice targets (side 160: duplicates and equidistant neighbours everywhere; or 600 000 lattice points
    each present twice, at original indices i and i + 600 000) against queries at lattice and half-integer positions, each
    equidistant to several targets.  The lowest-index rule holds through the grid kernel's tie pass (counter 1)."""
    side = 160
    if targets == "lattice":
        t = lattice_cloud(61, 1, 1_200_000, side=side)
    else:
        h = lattice_cloud(62, 1, 600_000, side=side)
        t = np.ascontiguousarray(np.concatenate([h, h], 1))
    rng = np.random.default_rng(63)
    q = (rng.integers(0, side, (1, QUERIES, 3)) + 0.5 * rng.integers(0, 2, (1, QUERIES, 3))).astype(np.float32)
    got, st, launched = traced(q, t, cuda, False)
    ran(launched, f"{P2}16,false>")
    assert st[2] > 0 and st[1] > 0, st
    ref, _ = run(q, t, cuda, "0")
    same(got, ref, f"{targets} vs exhaustive")
    secs = oracle_samples(q, t, got, 64)
    print(f"ties, {targets}: oracle samples {secs:.2f} s")


# ------------------------------------------------------------------------------------------------------------------ batches
@pytest.fixture(scope="module")
def batch_clouds():
    """9 cloud pairs of 40 000 queries x 600 000 targets (150 superblocks: SBR = 8), one scene each, each scaled and moved
    to its own extent; cloud 1 is in georeferenced coordinates (x ~ 5e5, y ~ 5e6, where float32 spacing is 0.5: exact
    distance ties are common)."""
    from genpc_b200.synthetic import lidar_scene_pair

    qs, ts = [], []
    for c in range(9):
        a, b = (x.numpy() for x in lidar_scene_pair(600_000, 40 + c))
        if c == 1:
            scale, off = 1.0, np.array([5.0e5, 5.0e6, 0.0])
        else:
            scale, off = 0.25 + 0.5 * c, np.array([30.0 * c, -20.0 * c, 0.5 * c])
        ts.append((a * scale + off).astype(np.float32))
        qs.append((b[:40000] * scale + off).astype(np.float32))
    return np.stack(qs), np.stack(ts)


@pytest.mark.parametrize("B", [2, 8])
def test_grid_scan_batches(cuda, batch_clouds, B):
    """B = 2 and B = 8 (the grid path's largest batch): bounding boxes and Hilbert keys per cloud, the key / value scratch reused
    cloud by cloud, one grid row per cloud."""
    q, t = (np.ascontiguousarray(x[:B]) for x in batch_clouds)
    got, st, launched = traced(q, t, cuda, False)
    for key in (f"{P2}8,false>", f"{P2}1,false>"):
        assert all(g[1] == B for g in ran(launched, key)), (key, launched[key])
    assert st[2] > 0, st
    ref, _ = run(q, t, cuda, "0")
    same(got, ref, f"B = {B} vs exhaustive")
    secs = oracle_samples(q, t, got, B)
    print(f"B = {B}: oracle samples {secs:.2f} s")


def test_nine_clouds_take_the_exhaustive_kernels(cuda, batch_clouds):
    """B = 9: the grid path sorts cloud by cloud and stops at 8 clouds; these clouds are too large for the one-CTA pruned scan."""
    q, t = batch_clouds
    got, st, launched = traced(q, t, cuda, False)
    no_grid_scan(launched)
    assert st[2] == 0, st
    secs = oracle_samples(q, t, got, 9)
    print(f"B = 9: oracle samples {secs:.2f} s")


# ------------------------------------------------------------------------------------------------------------- path limits
@pytest.mark.parametrize("layout,hand_back", [("lifted", False), ("shell", True)])
def test_probe_decides_at_16_superblock_registers(cuda, scene, layout, hand_back):
    """The probe (nn_prune2_kernel<16, true>) on 1.2M targets against 50 000 queries.
    lifted: the scene's targets, the queries lifted 1000 m.  The clouds do not overlap, yet every lifted query's nearest
    targets are the highest scene points below it, which the box bounds find at once (on a B200: 100 857 blocks walked by
    39 063 query groups).  The probe keeps the pruned scan, whose bounds here work on squared distances near 1e6.
    shell: targets on the unit sphere, queries within 1e-5 of its centre.  Every target is about equally far from every
    query, so a group would open nearly every block: the probe hands the pair to the exhaustive kernels and no real query
    group runs."""
    a, b = scene
    if layout == "lifted":
        t = a[None, :1_200_000]
        q = b[None, :QUERIES].copy()
        q[..., 2] += np.float32(1000)
    else:
        rng = np.random.default_rng(72)
        v = rng.standard_normal((1, 1_200_000, 3))
        t = (v / np.linalg.norm(v, axis=-1, keepdims=True)).astype(np.float32)
        q = ((rng.random((1, QUERIES, 3)) * 2 - 1) * 1e-5).astype(np.float32)
    got, st, launched = traced(q, t, cuda, False)
    ran(launched, f"{P2}16,true>")
    assert (st[2] == 0) == hand_back, st
    if not hand_back:
        ran(launched, f"{P2}16,false>")
    ref, _ = run(q, t, cuda, "0")
    same(got, ref, f"{layout} vs exhaustive")
    secs = oracle_samples(q, t, got, 70)
    print(f"probe, {layout}: oracle samples {secs:.2f} s")


def test_targets_past_the_grid_limit_take_the_exhaustive_kernels(cuda, scene):
    """GR_MAX_N + 1 targets: 513 superblocks do not fit the 9-bit id, the shape rule sends the pair to the exhaustive kernels."""
    a, b = scene
    q, t = b[None, :4096], a[None]
    assert superblocks(t.shape[1]) == 513
    got, st, launched = traced(q, t, cuda, False)
    no_grid_scan(launched)
    assert st[2] == 0, st
    secs = oracle_samples(q, t, got, 71)
    print(f"4096 x {t.shape[1]}: oracle samples {secs:.2f} s")
