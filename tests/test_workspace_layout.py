"""Workspace bounds of the pruned scans.  Every call runs on a workspace of exactly the size the library reports, placed inside a
larger buffer of sentinel bytes so that it starts 8 bytes past a 256-byte boundary: the start that needs the largest pad before
the pruned scan's extras (EMD asks for a 16-byte aligned workspace: 16 bytes past a boundary there).  The call must give what it
gives on a freshly allocated workspace, bit for bit, leave every sentinel byte outside its workspace as it was, and run the
pruned kernels.  A workspace 8 bytes short must keep the call on the exhaustive kernels (include/genpc_b200.h), with the same
results.  Covered: the Chamfer pruned scan from device and from host memory, the two-level grid scan with its probe at
1 048 576 x 1 048 576, the pruned registration loop and the pruned EMD Bid."""
import numpy as np
import pytest
import torch

from test_dispatch_paths import launched_kernels
from util import shape_cloud

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5
MARGIN = 4096


def placed(nbytes, dev, skew):
    """nbytes of workspace starting `skew` bytes past a 256-byte boundary inside a sentinel-filled buffer -> (workspace,
    check that no byte outside it changed)."""
    buf = torch.full((nbytes + 2 * MARGIN,), SENTINEL, dtype=torch.uint8, device=dev)
    off = MARGIN + (skew - buf.data_ptr()) % 256
    ws = buf[off:off + nbytes]
    assert ws.data_ptr() % 256 == skew

    def untouched():
        torch.cuda.synchronize()
        for part, where in ((buf[:off], "before"), (buf[off + nbytes:], "after")):
            bad = (part != SENTINEL).nonzero().flatten()
            assert bad.numel() == 0, f"{bad.numel()} sentinel bytes {where} the workspace changed"
    return ws, untouched


def same(got, exp, tag):
    for k, (g, e) in enumerate(zip(got, exp)):
        assert np.array_equal(g.view(np.int32), e.view(np.int32)), f"{tag}: output {k}: {(g.view(np.int32) != e.view(np.int32)).sum()} differ"


def check_bounds(dev, nbytes, call, pruned, skew=8):
    """call(workspace, nbytes) -> list of float32 / int32 arrays.  pruned: kernel keys (prefixes) of the pruned path."""
    fresh = call(torch.empty(nbytes, dtype=torch.uint8, device=dev), nbytes)
    for size in (nbytes, nbytes - 8):
        ws, untouched = placed(size, dev, skew)
        got, ks = launched_kernels(lambda: call(ws, size))
        untouched()
        same(got, fresh, f"workspace of {size} bytes")
        names = {k for k, _, _ in ks}
        for key in pruned:
            hit = sorted(k for k in names if k.startswith(key))
            if size == nbytes:
                assert hit, f"{key} did not run; launched: {sorted(names)}"
            else:
                assert not hit, f"a workspace 8 bytes short ran {hit}"


def chamfer_outputs(B, N, M, dev):
    return (torch.empty(B, N, device=dev), torch.empty(B, M, device=dev), torch.empty(B, N, dtype=torch.int32, device=dev),
            torch.empty(B, M, dtype=torch.int32, device=dev))


def chamfer_call(a, b, host=False):
    from genpc_b200 import _lib
    from genpc_b200.chamfer_3D import _feed

    B, N, M = a.shape[0], a.shape[1], b.shape[1]
    dev = torch.device("cuda:0")
    if host:
        ha, hb = torch.from_numpy(a).pin_memory(), torch.from_numpy(b).pin_memory()
        xa, xb = torch.empty(B, N, 3, device=dev), torch.empty(B, M, 3, device=dev)
    else:
        xa, xb = torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev)

    def call(ws, nbytes):
        out = chamfer_outputs(B, N, M, dev)
        o = [_lib.ptr(t) for t in out]
        L, stream = _lib.lib(), _lib.current_stream(dev)
        if host:
            xa.zero_(), xb.zero_()
            rc = L.genpc_chamfer_forward_host(_feed(dev), _lib.ptr(ha), _lib.ptr(hb), _lib.ptr(xa), _lib.ptr(xb), *o, B, N, M, 6,
                                              _lib.ptr(ws), nbytes, stream)
        else:
            rc = L.genpc_chamfer_forward(_lib.ptr(xa), _lib.ptr(xb), *o, B, N, M, _lib.ptr(ws), nbytes, stream)
        _lib.check(rc, "chamfer forward")
        return [t.cpu().numpy() for t in out]
    return call


@pytest.mark.parametrize("host", [False, True])
def test_chamfer_pruned_scan_stays_inside_its_workspace(cuda, host):
    """BASELINE C2's shape (32 x 2048 x 16384): Hilbert sort and pruned scan, device-resident and host-fed in two chunks."""
    from genpc_b200 import _lib

    B, N, M = 32, 2048, 16384
    L = _lib.lib()
    assert L.genpc_chamfer_scan_kind(B, N, M) == 1
    a, b = shape_cloud(11, B, N), shape_cloud(12, B, M)
    check_bounds(cuda, L.genpc_chamfer_workspace_bytes(B, N, M), chamfer_call(a, b, host),
                 ("genpc::nn_bin_sort_kernel<", "genpc::nn_prune_kernel<"))


def test_grid_scan_stays_inside_its_workspace(cuda):
    """1 048 576 x 1 048 576 scene clouds: the multi-CTA sort (cub's radix sort scratch last in the workspace), the probe and
    the two-level scan."""
    from genpc_b200 import _lib
    from genpc_b200.synthetic import lidar_scene_pair

    n = 1 << 20
    L = _lib.lib()
    assert L.genpc_chamfer_scan_kind(1, n, n) == 2
    a, b = lidar_scene_pair(n, 3)
    check_bounds(cuda, L.genpc_chamfer_workspace_bytes(1, n, n), chamfer_call(a.numpy()[None], b.numpy()[None]),
                 ("genpc::grid_key_kernel", "genpc::nn_prune2_kernel<8,true>", "genpc::nn_prune2_kernel<8,false>"))


def test_pruned_registration_stays_inside_its_workspace(cuda):
    """Four clouds, one start each (genpc_register_workspace_bytes sizes for that case), two iterations of the pruned loop."""
    from genpc_b200 import _lib
    from genpc_b200.optim_registration.diff_obj_pose import RegistrationBatch
    from test_registration import make_pair

    C, nc, nr, iters = 4, 6000, 4096, 2
    pairs = [make_pair(60 + c, nc, nr) for c in range(C)]
    V = torch.from_numpy(np.stack([p[0] for p in pairs])).to(cuda)
    Rf = torch.from_numpy(np.stack([p[1] for p in pairs])).to(cuda)

    def call(ws, nbytes):
        rb = RegistrationBatch(V, Rf, n_starts=1, lr=0.01, max_iters=iters)
        rb._ws, rb._ws_bytes = ws, nbytes
        rb.run(iters)
        return [t.cpu().numpy() for t in (rb.params, rb.adam_m, rb.adam_v, rb.losses())]

    with _lib.tunable(GENPC_REGISTER_PRUNE="1", GENPC_REGISTER_MODE="sym"):
        check_bounds(cuda, _lib.lib().genpc_register_workspace_bytes(C, nc, nr), call,
                     ("genpc::register_sims_kernel", "genpc::nn_prune_kernel<"))


def test_pruned_emd_stays_inside_its_workspace(cuda):
    """8 clouds of 4096 points: sort of the targets and the pruned Bid."""
    from genpc_b200 import _lib

    B, n = 8, 4096
    rng = np.random.default_rng(5)
    x1 = torch.from_numpy(rng.random((B, n, 3), dtype=np.float32)).to(cuda)
    x2 = torch.from_numpy(rng.random((B, n, 3), dtype=np.float32)).to(cuda)
    L = _lib.lib()

    def call(ws, nbytes):
        f = lambda *s: torch.zeros(*s, device=cuda)                       # noqa: E731
        i = lambda *s: torch.zeros(*s, dtype=torch.int32, device=cuda)    # noqa: E731
        dist, assignment, price, assignment_inv, bid = f(B, n), i(B, n), f(B, n), i(B, n), i(B, n)
        bufs = (dist, assignment, price, assignment_inv, bid, f(B, n), f(B, n), i(B * n), i(1024), i(B * n))
        rc = L.genpc_emd_forward(_lib.ptr(x1), _lib.ptr(x2), *[_lib.ptr(t) for t in bufs], B, n, n, 0.005, 50, _lib.ptr(ws), nbytes,
                                 _lib.current_stream(cuda))
        _lib.check(rc, "genpc_emd_forward")
        return [t.cpu().numpy() for t in (dist, assignment)]

    check_bounds(cuda, L.genpc_emd_workspace_bytes_n(B, n), call, ("genpc::nn_bin_sort_kernel<", "genpc::emd_auction_kernel<4,3>"),
                 skew=16)
