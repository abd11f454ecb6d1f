"""Per-lane culling in the pruned Chamfer walk (csrc/nn_prune.cuh, pr_visit_block): a block is fetched only when some query of
the warp is within its box, and an 8-target chunk is evaluated only when some query is within the chunk's box.  A wrong skip
changes a distance or, on exact ties, an index, so every case is compared bit for bit with the exhaustive kernels
(GENPC_CHAMFER_PRUNE=0) and, where it is quick, with the oracle."""
import numpy as np
import pytest

import oracle
from test_chamfer_prune import run, same
from util import shape_cloud

pytestmark = pytest.mark.gpu


def test_c2_batch_skips_chunks_and_matches_the_exhaustive_scan(cuda):
    """BASELINE C2: the same bits as the exhaustive scan, and the counters show that chunks inside walked blocks were skipped."""
    from genpc_b200.synthetic import pcn_batch

    part, comp = pcn_batch(0, 32, 2048, 16384)
    got, st = run(part, comp, cuda)
    ref, _ = run(part, comp, cuda, prune="0")
    same(got, ref, "C2 vs exhaustive")
    walked, chunks = int(st[0]), int(st[3])
    print("C2: %d blocks walked, %d of their %d chunks evaluated (%.1f %%), %.1f chunks per query group" %
          (walked, chunks, 8 * walked, 100.0 * chunks / (8 * walked), chunks / st[2]))
    assert 0 < chunks < 8 * walked, st


@pytest.mark.parametrize("coop", ["0", "1"])
@pytest.mark.parametrize("B,N,M", [(3, 2045, 9001), (2, 1031, 4099), (1, 777, 5003), (4, 4093, 4101)])
def test_sizes_off_the_chunk_and_block_grid(cuda, B, N, M, coop):
    """Clouds whose sizes are not multiples of 8 or 64: the last block holds NaN padding and chunks that are padding only
    (box +inf / -inf); both walk kernels (the cooperative one forced on and off)."""
    from genpc_b200 import _lib

    a, b = shape_cloud(N + B, B, N), shape_cloud(M + 11, B, M)
    with _lib.tunable(GENPC_PRUNE_COOP=coop):
        got, st = run(a, b, cuda)
    ref, _ = run(a, b, cuda, prune="0")
    same(got, ref, f"{B}x{N}x{M} coop={coop} vs exhaustive")
    if B * N * M <= 4e7:
        same(got, oracle.chamfer_forward(a, b), f"{B}x{N}x{M} coop={coop} vs oracle")
    assert st[2] > 0 and 0 < st[3] <= 8 * st[0], st


@pytest.mark.parametrize("coop", ["0", "1"])
def test_equal_distance_targets_in_different_chunks_of_one_block(cuda, coop):
    """Every lattice point is a target 12 times over, in shuffled order: the copies sort next to each other (one Hilbert cell) and
    so span two or three chunks of a block, all at the same distance from a query.  Queries sit on lattice points and halfway
    between them (equidistant from the copies of two to eight points).  The lowest original index wins only if no chunk
    holding a copy is skipped."""
    from genpc_b200 import _lib

    rng = np.random.default_rng(12)
    side = 8
    grid = np.stack(np.meshgrid(*[np.arange(side)] * 3, indexing="ij"), -1).reshape(-1, 3)
    tgt = np.repeat(grid, 12, 0)[rng.permutation(len(grid) * 12)].astype(np.float32)[None]      # 6144 targets
    q = rng.integers(0, side * 2 - 1, size=(1, 3000, 3)).astype(np.float32) * np.float32(0.5)  # lattice and half-lattice
    for a, b, tag in ((q, tgt, "queries -> copies"), (tgt, q, "copies -> queries")):
        with _lib.tunable(GENPC_PRUNE_COOP=coop):
            got, st = run(a, b, cuda)
        same(got, oracle.chamfer_forward(a, b), f"{tag} coop={coop} vs oracle")
        ref, _ = run(a, b, cuda, prune="0")
        same(got, ref, f"{tag} coop={coop} vs exhaustive")
        assert st[2] > 0 and st[1] > 0, st   # the pruned kernels ran, and ties sent groups through the second pass
