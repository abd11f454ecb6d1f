"""Sequences of Chamfer calls on the cached step workspace (chamfer_3D.step_workspace), each call against references that do not
depend on the cache.

Every device-resident Chamfer call (chamfer_3DDist, Completionloss's Chamfer forms, ragged or not, get_loss_from_host,
GraphedLossStep) goes through chamfer_3D.forward_fused, which takes its scratch from a process-wide cache keyed by (device,
stream, B, N, M): at most 16 entries, the oldest dropped first.  An entry is "armed" when the last call left every packed word
all-ones, and the next call then skips the memset; a captured graph bakes the entry's pointers in.  So whether a call is right
depends on what earlier calls left behind.  The schedules below change the data, the knobs, the path, the stream and the number
of live keys between calls of one shape, and compare after every call:
- dist / idx bit for bit with oracle.chamfer_forward (ragged batches: per pair, test_chamfer_ragged.expected);
- the loss within 1e-6 relative of a float64 mean over the oracle's distances, the gradients within 1e-5 of the largest
  oracle.chamfer_backward gradient (ragged batches: test_chamfer_ragged.loss_oracle);
- for the 50 000 x 524 289 grid-scan shape, where a full oracle run is too slow: an uncached exhaustive call
  (GENPC_CHAMFER_PRUNE=0) bit for bit, plus 2048 sampled queries per direction against the oracle.
Before comparing, each call asserts which path ran (pruned-scan counters or the profiler's kernel list), so a moved threshold
fails instead of quietly testing another path."""
import contextlib
import weakref

import numpy as np
import pytest
import torch

import oracle
from test_chamfer_large_clouds import oracle_samples
from test_chamfer_ragged import expected, lengths_for, loss_oracle
from test_dispatch_paths import launched_kernels
from util import rand_cloud, shape_cloud

pytestmark = pytest.mark.gpu

C2 = (32, 2048, 16384)          # BASELINE C2: Hilbert-sorted pruned scan, cooperative kernel on a side stream
GRID = (1, 50000, 524289)       # two-level pruned scan by default (129 superblocks: nn_prune2_kernel<8>)
L1, L2 = ("cd_l1", True, 0.5, 0.5), ("cd_l2", False, 1.0, 1.0)   # Completionloss form, use_sqrt, w1, w2 of get_loss


@contextlib.contextmanager
def prune_counters(dev):
    """The pruned scans' counters (genpc_chamfer_prune_stats) for the duration of the block; [2] > 0: a pruned scan did the
    work.  Launches captured into a graph inside the block keep counting on replay while the tensor lives."""
    from genpc_b200 import _lib

    stats = torch.zeros(4, dtype=torch.int32, device=dev)
    _lib.lib().genpc_chamfer_prune_stats(_lib.ptr(stats))
    try:
        yield stats
    finally:
        _lib.lib().genpc_chamfer_prune_stats(None)


def pruned(stats):
    """Read and reset the counters -> True if a pruned scan did the work since the last reset."""
    torch.cuda.synchronize()
    did = int(stats[2]) > 0
    stats.zero_()
    return did


def np_out(ts):
    return [t.detach().cpu().numpy() for t in ts]


def assert_bits(got, exp, tag, keep=None):
    """dist1, dist2, idx1, idx2 bit for bit (keep: optional masks of the entries to compare, for dist1 / idx1 and dist2 / idx2)."""
    for k, (g, e, name) in enumerate(zip(got, exp, ("dist1", "dist2", "idx1", "idx2"))):
        g, e = np.asarray(g), np.asarray(e)
        assert g.dtype == e.dtype and g.shape == e.shape, (tag, name, g.dtype, e.dtype, g.shape, e.shape)
        if keep is not None:
            g, e = g[keep[k % 2]], e[keep[k % 2]]
        bad = g.view(np.int32) != e.view(np.int32)
        assert not bad.any(), f"{tag}: {name} differs in {bad.sum()} of {bad.size} entries"


def loss_expect(a, b, e, cfg):
    """float64 loss of an equal-size batch over the oracle's (or a reference's) distances e, and the float64 gradients of it
    (oracle.chamfer_backward with graddist = w / (B * n) (* 0.5 / sqrt d))."""
    _, use_sqrt, w1, w2 = cfg
    B, N, M = a.shape[0], a.shape[1], b.shape[1]
    d1, d2 = e[0].astype(np.float64), e[1].astype(np.float64)
    f = np.sqrt if use_sqrt else (lambda d: d)
    loss = w1 * f(d1).mean() + w2 * f(d2).mean()
    s1 = np.full(d1.shape, w1 / (B * N)) * (0.5 / np.sqrt(d1) if use_sqrt else 1.0)
    s2 = np.full(d2.shape, w2 / (B * M)) * (0.5 / np.sqrt(d2) if use_sqrt else 1.0)
    g1, g2 = oracle.chamfer_backward(a, b, s1.astype(np.float32), s2.astype(np.float32), e[2], e[3])
    return loss, g1, g2


def assert_loss(tag, loss, ga, gb, exp):
    want, e1, e2 = exp
    assert abs(loss - want) <= 1e-6 * abs(want), (tag, loss, want)
    for g, e, name in ((ga, e1, "grad gen"), (gb, e2, "grad gt")):
        err = np.abs(g - e).max()
        assert err <= 1e-5 * np.abs(e).max() + 1e-12, (tag, name, err, np.abs(e).max())


def loss_step(cl, a, b, dev, len1=None, len2=None):
    """get_loss + backward on fresh leaves -> (dist1, dist2, idx1, idx2 of the call, loss, grad gen, grad gt), numpy."""
    ta = torch.from_numpy(a).to(dev).requires_grad_(True)
    tb = torch.from_numpy(b).to(dev).requires_grad_(True)
    loss = cl.get_loss(ta, tb, len1, len2)
    out = np_out(loss.grad_fn.saved_tensors[2:])   # (xyz1, xyz2, dist1, dist2, idx1, idx2) of the fused call
    loss.backward()
    return out, float(loss), ta.grad.cpu().numpy(), tb.grad.cpu().numpy()


def check_equal_size(tag, cl_cfg, a, b, res, e=None):
    """A get_loss call of an equal-size batch against the oracle."""
    out, loss, ga, gb = res
    e = oracle.chamfer_forward(a, b) if e is None else e
    assert_bits(out, e, tag)
    assert_loss(tag, loss, ga, gb, loss_expect(a, b, e, cl_cfg))
    return e


def uncached_exhaustive(a, b, dev):
    """chamfer_3D.forward (a fresh workspace per call, no cache) with the pruned scans switched off."""
    from genpc_b200 import _lib, chamfer_3D

    B, N, M = a.shape[0], a.shape[1], b.shape[1]
    ta, tb = torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev)
    out = [torch.empty(B, N, device=dev), torch.empty(B, M, device=dev),
           torch.empty(B, N, dtype=torch.int32, device=dev), torch.empty(B, M, dtype=torch.int32, device=dev)]
    with _lib.tunable(GENPC_CHAMFER_PRUNE="0"):
        chamfer_3D.forward(ta, tb, *out)
    return np_out(out)


# ------------------------------------------------------------------------------------------------------------ inputs
def c2_inputs():
    """C2 inputs in schedule order: clean, far apart, one collapsed blob, one NaN point (eager only), clean again (other
    shapes).  The pruned scan hands the middle three back to the exhaustive kernels (overlap test, size test, range check)."""
    from genpc_b200.synthetic import pcn_batch

    part, comp = pcn_batch(0, *C2)
    part2, comp2 = pcn_batch(1, *C2)
    rng = np.random.default_rng(90)
    blob = (np.float32(0.1) + rng.random(part.shape, dtype=np.float32) * np.float32(1e-3)).astype(np.float32)
    nan = part2.copy()
    nan[3, 100] = np.nan
    return [("clean", part, comp, True), ("far apart", part, (comp + np.float32(1000)).astype(np.float32), False),
            ("blob", blob, comp, False), ("nan", nan, comp2, False), ("clean again", part2, comp2, True)]


def grid_inputs():
    """GRID inputs in schedule order: 50 000 scene queries against a 524 289-point scene, a spherical shell around queries at
    its centre (the probe hands the pair to the exhaustive kernels, test_probe_decides_at_16_superblock_registers), one NaN
    query (eager only: the range check hands back), other scene queries again."""
    from genpc_b200.synthetic import lidar_scene_pair

    B, N, M = GRID
    a, b = (x.numpy() for x in lidar_scene_pair(M, 0))
    rng = np.random.default_rng(72)
    v = rng.standard_normal((1, M, 3))
    shell = (v / np.linalg.norm(v, axis=-1, keepdims=True)).astype(np.float32)
    centre = ((rng.random((1, N, 3)) * 2 - 1) * 1e-5).astype(np.float32)
    q1, q2 = np.ascontiguousarray(b[None, :N]), np.ascontiguousarray(b[None, N:2 * N])
    nan = q1.copy()
    nan[0, 1234, 1] = np.nan
    t = np.ascontiguousarray(a[None])
    return [("clean", q1, t, True), ("shell", centre, shell, False), ("nan", nan, t, False), ("clean again", q2, t, True)]


def check_nan_call(tag, cfg, a, b, res, dev, grid):
    """A call with one NaN point: bit for bit the uncached exhaustive kernels; the oracle on every entry that never met the
    poisoned point (its own row, and the rows whose clean nearest neighbour it was); the loss is the float64 mean over the
    exhaustive distances, which is not finite (the poisoned row's distance is not)."""
    out, loss, _, _ = res
    ref = uncached_exhaustive(a, b, dev)
    assert_bits(out, ref, tag + " vs exhaustive")
    _, use_sqrt, w1, w2 = cfg
    f = np.sqrt if use_sqrt else (lambda d: d)
    with np.errstate(invalid="ignore"):
        want = w1 * f(ref[0].astype(np.float64)).mean() + w2 * f(ref[1].astype(np.float64)).mean()
    assert not np.isfinite(want) and (loss == want or (np.isnan(loss) and np.isnan(want))), (tag, loss, want)
    if grid:
        return   # (the exhaustive reference above; the other calls of the schedule check the grid kernels against the oracle)
    bad = np.argwhere(np.isnan(a).any(-1))
    assert len(bad) == 1
    c, j = bad[0]
    clean = a.copy()
    clean[c, j] = 0.0
    e = oracle.chamfer_forward(clean, b)
    keep1 = np.ones(a.shape[:2], bool)
    keep1[c, j] = False
    keep2 = np.ones(b.shape[:2], bool)
    keep2[c] &= e[3][c] != j
    # the clean cloud's row j and the columns whose nearest it was are the poisoned entries; the rest keep the oracle's answer
    assert_bits(out, e, tag + " vs oracle (unpoisoned entries)", keep=(keep1, keep2))


def check_grid_call(tag, cfg, a, b, res, dev, seed):
    out, loss, ga, gb = res
    ref = uncached_exhaustive(a, b, dev)
    assert_bits(out, ref, tag + " vs exhaustive")
    oracle_samples(a, b, out, seed)
    assert_loss(tag, loss, ga, gb, loss_expect(a, b, ref, cfg))
    return ref


# -------------------------------------------------------------------------------------- 1. data switches the path
@pytest.mark.parametrize("shape", ["c2", "grid"])
def test_data_switches_the_path_on_one_armed_entry(cuda, shape):
    """One shape, one cached entry: clean -> inputs the pruned scan hands back -> clean again, eagerly through Completionloss,
    then through one GraphedLossStep with the inputs written in place, every replay against the oracle."""
    from genpc_b200 import _lib
    from genpc_b200.utils.loss_util import Completionloss, GraphedLossStep

    B, N, M = C2 if shape == "c2" else GRID
    assert _lib.lib().genpc_chamfer_scan_kind(B, N, M) == (1 if shape == "c2" else 2)
    cfg = L2 if shape == "c2" else L1
    inputs = c2_inputs() if shape == "c2" else grid_inputs()
    cl = Completionloss(cfg[0])
    refs = {}   # the references of the eager calls (oracle, or exhaustive + sampled oracle), reused for the replays
    with prune_counters(cuda) as stats:
        for k, (name, a, b, prunes) in enumerate(inputs):
            res = loss_step(cl, a, b, cuda)
            assert pruned(stats) == prunes, (shape, name)
            tag = f"{shape} eager {name}"
            if name == "nan":
                check_nan_call(tag, cfg, a, b, res, cuda, shape == "grid")
            elif shape == "c2":
                refs[name] = check_equal_size(tag, cfg, a, b, res)
            else:
                refs[name] = check_grid_call(tag, cfg, a, b, res, cuda, k)
        step = GraphedLossStep(cl, torch.from_numpy(inputs[0][1]).to(cuda), torch.from_numpy(inputs[0][2]).to(cuda))
        for k, (name, a, b, prunes) in enumerate(inputs):
            if name == "nan":
                continue
            step.gen.data.copy_(torch.from_numpy(a).to(cuda))
            step.gt.data.copy_(torch.from_numpy(b).to(cuda))
            stats.zero_()
            loss, ga, gb = step()
            assert pruned(stats) == prunes, (shape, "graph", name)
            res_loss, res_ga, res_gb = float(loss), ga.cpu().numpy(), gb.cpu().numpy()
            assert_loss(f"{shape} graph {name}", res_loss, res_ga, res_gb, loss_expect(a, b, refs[name], cfg))


# ---------------------------------------------------------------------------------------------------- 2. knob flips
def _kernels_of(fn):
    out, ks = launched_kernels(fn)
    return out, {k for k, _, _ in ks}


@pytest.mark.parametrize("knob", ["GENPC_CHAMFER_MODE", "GENPC_SYM_BALANCED"])
def test_knob_flips_between_same_shape_calls(cuda, knob):
    """4 x 2600 x 700 (two rows per thread), new clouds on every call, the knob flipped between calls of one shape on one
    stream.  GENPC_CHAMFER_MODE=scan takes the per-direction scan (nn_scan_kernel + nn_unpack_kernel), the default the symmetric
    one; GENPC_SYM_BALANCED=0 / 1 the item grid / the balanced grid of the symmetric scan.  After a per-direction call the next
    symmetric call skips the memset, so the per-direction path must leave the packed words all-ones, and its loss kernel must
    leave the epilogue's ticket in the shared loss workspace alone."""
    from genpc_b200 import _lib
    from genpc_b200.utils.loss_util import Completionloss

    B, N, M = 4, 2600, 700
    values = [None, "scan", None, "scan", None] if knob == "GENPC_CHAMFER_MODE" else ["0", "1", "0", "1"]
    kernel = {"scan": "genpc::nn_scan_kernel<2>", None: "genpc::nn_sym_balanced_kernel<4>",
              "0": "genpc::nn_sym_kernel<4>", "1": "genpc::nn_sym_balanced_kernel<4>"}
    for k, cfg in enumerate([L1, L2]):
        cl = Completionloss(cfg[0])
        for call, v in enumerate(values):
            a, b = shape_cloud(500 + 10 * k + call, B, N), rand_cloud(600 + 10 * k + call, B, M, 0.8, -0.4)
            with _lib.tunable(**{knob: v}):
                res, ks = _kernels_of(lambda: loss_step(cl, a, b, cuda))
            assert kernel[v] in ks, (knob, v, sorted(ks))
            assert ("genpc::nn_unpack_kernel" in ks) == (v == "scan"), (knob, v, sorted(ks))
            check_equal_size(f"{knob}={v}, {cfg[0]}, call {call}", cfg, a, b, res)


def test_pruned_scan_knob_flips_at_c2(cuda):
    """C2 on one stream: the cooperative kernel forbidden / forced, sort-cluster layouts, the pruned scan switched off (a
    workspace of another size: the entry is replaced) and back on; new clouds on every call."""
    from genpc_b200 import _lib
    from genpc_b200.synthetic import pcn_batch
    from genpc_b200.utils.loss_util import Completionloss

    schedule = [{}, {"GENPC_PRUNE_COOP": "0"}, {"GENPC_PRUNE_COOP": "1"}, {"GENPC_SORT_CLUSTER": "m2"},
                {"GENPC_SORT_CLUSTER": "8"}, {"GENPC_CHAMFER_PRUNE": "0"}, {}, {"GENPC_CHAMFER_PRUNE": "0"}, {"GENPC_PRUNE_COOP": "0"}]
    cl = Completionloss(L2[0])
    with prune_counters(cuda) as stats:
        for call, knobs in enumerate(schedule):
            a, b = pcn_batch(10 + call, *C2)
            with _lib.tunable(**knobs):
                res, ks = _kernels_of(lambda: loss_step(cl, a, b, cuda))
            prunes = knobs.get("GENPC_CHAMFER_PRUNE") != "0"
            assert pruned(stats) == prunes, (knobs, sorted(ks))
            coop = any(k.startswith("genpc::nn_prune_coop_kernel<") for k in ks)
            assert coop == (prunes and knobs.get("GENPC_PRUNE_COOP") != "0"), (knobs, sorted(ks))
            if knobs.get("GENPC_SORT_CLUSTER") == "8":
                assert "genpc::nn_bin_sort_kernel<8>" in ks, sorted(ks)
            check_equal_size(f"C2 {knobs} call {call}", L2, a, b, res)


# ------------------------------------------------------------------------------------------------------- 3. eviction
def _other_keys(dev, count, first):
    """`count` distinct cache keys on the current stream (equal-size shapes and ragged strides no other test uses), every call
    against the oracle."""
    from genpc_b200.loss_functions import chamfer_3DDist

    rng = np.random.default_rng(first)
    for k in range(count):
        B, N, M = 2, first + 3 * k, first + 3 * k + 101
        a, b = shape_cloud(first + k, B, N), rand_cloud(first + 50 + k, B, M, 0.8, -0.4)
        if k % 2:
            l1, l2 = lengths_for(rng, B, N), lengths_for(rng, B, M)
            out = chamfer_3DDist()(torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev), torch.from_numpy(l1).to(dev),
                                   torch.from_numpy(l2).to(dev))
            assert_bits(np_out(out), expected(a, b, l1, l2), f"key {k} ragged")
        else:
            out = chamfer_3DDist()(torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev))
            assert_bits(np_out(out), oracle.chamfer_forward(a, b), f"key {k}")


def _key(dev, stream, B, N, M):
    return (dev.index, stream.cuda_stream, B, N, M)


def test_more_keys_than_the_cache_holds_then_back(cuda):
    """Two shapes armed (one equal-size, one ragged), 17 other keys (the first two are dropped), then both shapes again with
    new clouds: fresh entries, right answers; the cache never holds more than 16 entries."""
    from genpc_b200 import chamfer_3D
    from genpc_b200.utils.loss_util import Completionloss

    cl = Completionloss(L1[0])
    rng = np.random.default_rng(3)
    shapes = [(3, 1500, 900, False), (5, 1100, 1700, True)]

    def calls(seed):
        for B, N, M, ragged in shapes:
            a, b = shape_cloud(seed + N, B, N), shape_cloud(seed + M, B, M)
            if ragged:
                l1, l2 = lengths_for(rng, B, N), lengths_for(rng, B, M)
                out, loss, ga, gb = loss_step(cl, a, b, cuda, torch.from_numpy(l1).to(cuda), torch.from_numpy(l2).to(cuda))
                assert_bits(out, expected(a, b, l1, l2), f"ragged {B}x{N}x{M}, seed {seed}")
                assert_loss(f"ragged {B}x{N}x{M}", loss, ga, gb, loss_oracle(a, b, l1, l2, *L1[1:]))
            else:
                check_equal_size(f"{B}x{N}x{M}, seed {seed}", L1, a, b, loss_step(cl, a, b, cuda))

    stream = torch.cuda.current_stream(cuda)
    for seed in (1, 2):
        calls(seed)
    refs = [weakref.ref(chamfer_3D._step_ws[_key(cuda, stream, *s[:3])]) for s in shapes]
    _other_keys(cuda, 17, 601)
    assert len(chamfer_3D._step_ws) <= 16
    assert all(_key(cuda, stream, *s[:3]) not in chamfer_3D._step_ws for s in shapes) and all(r() is None for r in refs)
    for seed in (3, 4):
        calls(seed)


@pytest.mark.parametrize("drop", ["eviction", "knob"])
def test_graph_owns_its_workspace(cuda, drop):
    """A GraphedLossStep's cache entry is dropped after the capture -- by 17 other keys on the default stream, or by a
    GENPC_CHAMFER_PRUNE flip and an eager call of the same shape on step.stream (a workspace of another size replaces the
    entry).  The entry must stay alive (the graph bakes its pointers in) BEFORE any replay; then a tensor of the same size
    allocated on step.stream keeps its contents through a replay with new clouds, and the replay matches the oracle."""
    from genpc_b200 import _lib, chamfer_3D
    from genpc_b200.utils.loss_util import Completionloss, GraphedLossStep

    B, N, M = 4, 2048, 4096
    cl = Completionloss(L1[0])
    step = GraphedLossStep(cl, torch.from_numpy(shape_cloud(1, B, N)).to(cuda), torch.from_numpy(shape_cloud(2, B, M)).to(cuda))
    key = _key(cuda, step.stream, B, N, M)
    ws = weakref.ref(chamfer_3D._step_ws[key])
    if drop == "eviction":
        _other_keys(cuda, 17, 701)
    else:
        a, b = shape_cloud(3, B, N), shape_cloud(4, B, M)
        with _lib.tunable(GENPC_CHAMFER_PRUNE="1"), prune_counters(cuda) as stats, torch.cuda.stream(step.stream):
            res = loss_step(cl, a, b, cuda)
            assert pruned(stats)
        check_equal_size("eager call on step.stream, pruned", L1, a, b, res)
    torch.cuda.synchronize()
    captured = ws()
    assert captured is not None, "the captured workspace was freed while the graph still uses it"
    assert chamfer_3D._step_ws.get(key) is not captured, "the cache still holds the captured entry: nothing was dropped"
    del captured
    with torch.cuda.stream(step.stream):
        sentinels = [torch.full((t.numel(),), 0x5A, dtype=torch.uint8, device=cuda) for t in (ws().packed, ws().loss)]
    torch.cuda.synchronize()
    for seed in (5, 7):
        a, b = shape_cloud(seed, B, N), shape_cloud(seed + 1, B, M)
        step.gen.data.copy_(torch.from_numpy(a).to(cuda))
        step.gt.data.copy_(torch.from_numpy(b).to(cuda))
        loss, ga, gb = step()
        torch.cuda.synchronize()
        assert_loss(f"replay after {drop}, seed {seed}", float(loss), ga.cpu().numpy(), gb.cpu().numpy(),
                    loss_expect(a, b, oracle.chamfer_forward(a, b), L1))
        assert all(bool((s == 0x5A).all()) for s in sentinels), "a replay wrote into memory the step does not own"


# ------------------------------------------------------------------------------------------ 4. mixed entries on one key
@pytest.mark.parametrize("shape", [C2, (3, 1500, 900)], ids=["c2", "3x1500x900"])
def test_mixed_entry_points_on_one_key(cuda, shape):
    """chamfer_3DDist (no loss), a fused Completionloss, a ragged Completionloss and get_loss_from_host, alternating on one
    (device, stream, shape) entry, new clouds on every call.  C2: the equal-size calls take the pruned scan (the host-fed one
    chunk by chunk), the ragged call the exhaustive one on the same workspace."""
    from genpc_b200.loss_functions import chamfer_3DDist
    from genpc_b200.utils.loss_util import Completionloss

    B, N, M = shape
    big = shape == C2
    cl = Completionloss(L1[0])
    rng = np.random.default_rng(17)
    with prune_counters(cuda) as stats:
        for call in range(8):
            kind = ("dist", "loss", "ragged", "host")[call % 4]
            a, b = shape_cloud(800 + call, B, N), shape_cloud(900 + call, B, M)
            tag = f"{shape} call {call} {kind}"
            if kind == "dist":
                out = np_out(chamfer_3DDist()(torch.from_numpy(a).to(cuda), torch.from_numpy(b).to(cuda)))
                assert pruned(stats) == big, tag
                assert_bits(out, oracle.chamfer_forward(a, b), tag)
            elif kind == "loss":
                res = loss_step(cl, a, b, cuda)
                assert pruned(stats) == big, tag
                check_equal_size(tag, L1, a, b, res)
            elif kind == "ragged":
                l1, l2 = lengths_for(rng, B, N), lengths_for(rng, B, M)
                out, loss, ga, gb = loss_step(cl, a, b, cuda, torch.from_numpy(l1).to(cuda), torch.from_numpy(l2).to(cuda))
                assert not pruned(stats), tag
                assert_bits(out, expected(a, b, l1, l2), tag)
                assert_loss(tag, loss, ga, gb, loss_oracle(a, b, l1, l2, *L1[1:]))
            else:
                loss, ta, tb = cl.get_loss_from_host(torch.from_numpy(a).pin_memory(), torch.from_numpy(b).pin_memory(), cuda)
                out = np_out(loss.grad_fn.saved_tensors[2:])
                loss.backward()
                assert pruned(stats) == big, tag
                check_equal_size(tag, L1, a, b, (out, float(loss), ta.grad.cpu().numpy(), tb.grad.cpu().numpy()))


# -------------------------------------------------------------------------------------------- 5. streams and devices
def test_one_shape_on_two_streams_interleaved(cuda):
    """C2 on two streams (two cache entries, two cooperative side streams), four loss steps issued alternately with no
    synchronisation between them; each against the oracle afterwards."""
    from genpc_b200.synthetic import pcn_batch
    from genpc_b200.utils.loss_util import Completionloss

    cl = Completionloss(L2[0])
    streams = [torch.cuda.Stream(cuda), torch.cuda.Stream(cuda)]
    clouds = [pcn_batch(20 + k, *C2) for k in range(4)]
    leaves = [(torch.from_numpy(a).to(cuda).requires_grad_(True), torch.from_numpy(b).to(cuda).requires_grad_(True))
              for a, b in clouds]
    for s in streams:
        s.wait_stream(torch.cuda.current_stream(cuda))
    results = []
    with prune_counters(cuda) as stats:
        for k, (ta, tb) in enumerate(leaves):
            with torch.cuda.stream(streams[k % 2]):
                loss = cl.get_loss(ta, tb)
                saved = loss.grad_fn.saved_tensors[2:]
                loss.backward()
                results.append((loss.detach(), saved))
        torch.cuda.synchronize()
        assert int(stats[2]) == 4 * 32 * (2048 // 32 + 16384 // 32), stats   # every call took the pruned scan
    for k, ((a, b), (ta, tb), (loss, saved)) in enumerate(zip(clouds, leaves, results)):
        check_equal_size(f"stream {k % 2}, call {k}", L2, a, b, (np_out(saved), float(loss), ta.grad.cpu().numpy(),
                                                                 tb.grad.cpu().numpy()))


def test_tensors_on_another_device_than_the_current_one():
    """Tensors on cuda:1 while cuda:0 is current, alternating with the same shape on cuda:0 (one entry per device)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from genpc_b200.loss_functions import chamfer_3DDist
    from genpc_b200.utils.loss_util import Completionloss

    B, N, M = 3, 1500, 900
    cl = Completionloss(L1[0])
    torch.cuda.set_device(0)
    for call in range(4):
        dev = torch.device("cuda", (call + 1) % 2)
        a, b = shape_cloud(40 + call, B, N), shape_cloud(50 + call, B, M)
        assert torch.cuda.current_device() == 0
        check_equal_size(f"{dev} loss, call {call}", L1, a, b, loss_step(cl, a, b, dev))
        out = np_out(chamfer_3DDist()(torch.from_numpy(b).to(dev), torch.from_numpy(a).to(dev)))
        assert_bits(out, oracle.chamfer_forward(b, a), f"{dev} dist, call {call}")


def test_a_call_that_fails_its_checks_does_not_disturb_the_next(cuda):
    """Calls with bad lengths (floating point, wrong shape, another device type) in the middle of a sequence on one armed entry:
    they raise, and the next calls (equal-size and ragged) are right."""
    from genpc_b200 import _lib
    from genpc_b200.utils.loss_util import Completionloss

    B, N, M = 4, 1800, 1200
    cl = Completionloss(L2[0])
    rng = np.random.default_rng(9)
    bad = [torch.full((B,), 3.0, device=cuda), torch.full((B + 1,), N, dtype=torch.int32, device=cuda),
           torch.full((B,), N, dtype=torch.int32)]
    for call in range(6):
        a, b = shape_cloud(70 + call, B, N), shape_cloud(80 + call, B, M)
        check_equal_size(f"call {call}", L2, a, b, loss_step(cl, a, b, cuda))
        with pytest.raises(_lib.GenpcError):
            loss_step(cl, a, b, cuda, bad[call % 3], None)
        l1, l2 = lengths_for(rng, B, N), lengths_for(rng, B, M)
        out, loss, ga, gb = loss_step(cl, a, b, cuda, torch.from_numpy(l1).to(cuda), torch.from_numpy(l2).to(cuda))
        assert_bits(out, expected(a, b, l1, l2), f"ragged call {call}")
        assert_loss(f"ragged call {call}", loss, ga, gb, loss_oracle(a, b, l1, l2, *L2[1:]))
