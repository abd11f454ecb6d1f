"""CPU: the C-ABI library loads and exports every symbol include/*.h declares (no compute calls)."""
import ctypes
import glob
import os
import re

from conftest import ROOT


def declared_symbols():
    syms = set()
    for h in glob.glob(os.path.join(ROOT, "include", "*.h")):
        txt = re.sub(r"/\*.*?\*/", "", open(h).read(), flags=re.S)
        syms |= set(re.findall(r"\b(genpc_[a-z0-9_]+)\s*\(", txt))
    return sorted(syms)


def test_header_declares_something():
    assert "genpc_chamfer_forward" in declared_symbols()


def test_library_exports_every_declared_symbol():
    from genpc_b200.csrc import build

    so = build.build()
    L = ctypes.CDLL(so)
    missing = [s for s in declared_symbols() if not hasattr(L, s)]
    assert not missing, f"declared in include/ but not exported: {missing}"


def test_python_binding_table_matches_header():
    from genpc_b200 import _lib

    assert sorted(_lib._SIGNATURES) == declared_symbols()
    L = _lib.lib()
    assert L.genpc_version().decode().startswith("genpc_b200")
    assert L.genpc_chamfer_workspace_bytes(2, 3, 5) == (2 * 3 + 2 * 5) * 8 + 16


def test_no_cpu_fallback():
    import pytest
    import torch

    from genpc_b200 import _lib
    from genpc_b200.loss_functions import chamfer_3DDist

    with pytest.raises(_lib.GenpcError):
        chamfer_3DDist()(torch.rand(1, 4, 3), torch.rand(1, 5, 3))


def test_scan_selection_host_logic():
    """Which Chamfer scan the library would queue (host logic, no device): exhaustive for small batches, the Hilbert-sorted pruned
    scan from 2^30 evaluations, the two-level pruned scan for large clouds; the knob overrides; workspace sizes follow."""
    from genpc_b200 import _lib

    L = _lib.lib()
    kind = L.genpc_chamfer_scan_kind
    assert kind(32, 2048, 16384) == 1 and kind(32, 16384, 2048) == 1          # BASELINE C2: 2^30 evaluations
    assert kind(8, 8192, 8192) == 0 and kind(16, 8192, 8192) == 1
    assert kind(1, 71372, 16384) == 0                                         # C1: below 2^32 evaluations
    assert kind(1, 1000000, 1000000) == 2 and kind(9, 1000000, 1000000) == 0  # C5; the grid path sorts cloud by cloud (B <= 8)
    assert kind(8, 600000, 40000) == 2 and kind(9, 600000, 40000) == 0
    assert kind(1, 2097152, 2048) == 2 and kind(1, 2097152, 2047) == 0        # GR_MAX_N targets; from 2^32 evaluations
    assert kind(1, 2097153, 4096) == 0                                        # 513 superblocks: past the 9-bit superblock id
    assert kind(32, 512, 4096) == 0 and kind(4, 100, 37) == 0
    assert kind(1000, 1791, 1755) == 0                                        # the ICP scale search: clouds too small for the sort to pay
    assert kind(0, 5, 5) < 0
    base = lambda B, N, M: (B * N + B * M) * 8 + 16                           # noqa: E731
    assert L.genpc_chamfer_workspace_bytes(8, 8192, 8192) == base(8, 8192, 8192)
    assert L.genpc_chamfer_workspace_bytes(32, 2048, 16384) > base(32, 2048, 16384) + 32 * (2048 + 16384) * 16
    with _lib.tunable(GENPC_CHAMFER_PRUNE="0"):
        assert kind(32, 2048, 16384) == 0 and kind(1, 1000000, 1000000) == 0
        assert L.genpc_chamfer_workspace_bytes(32, 2048, 16384) == base(32, 2048, 16384)
    with _lib.tunable(GENPC_CHAMFER_PRUNE="1"):
        assert kind(2, 700, 1300) == 1 and kind(2, 40, 1300) == 0
    with _lib.tunable(GENPC_CHAMFER_PRUNE="2"):
        assert kind(2, 700, 1300) == 2
    assert L.genpc_emd_workspace_bytes_n(32, 8192) > L.genpc_emd_workspace_bytes(32) + 32 * 8192 * 16
    assert L.genpc_emd_workspace_bytes_n(1, 65536) == L.genpc_emd_workspace_bytes(1)   # beyond the pruned Bid's range


def test_sort_layout_host_logic():
    """Layout of the pruned scan's sort kernel (host logic, no device): clusters only for clouds of >= 8192 points, the largest
    cluster size whose grid is one wave of one CTA per SM, the mixed layout when one side is >= 4x smaller, knob overrides."""
    import ctypes

    from genpc_b200 import _lib

    L = _lib.lib()

    def layout(B, N, M, sms=148):
        mixed, grid = ctypes.c_int(-1), ctypes.c_int(-1)
        cs = L.genpc_chamfer_sort_layout(B, N, M, sms, ctypes.byref(mixed), ctypes.byref(grid))
        return cs, mixed.value, grid.value

    assert layout(32, 2048, 16384) == (3, 1, 129) == layout(32, 16384, 2048)      # BASELINE C2: 32 x 3 + 33 CTAs
    assert layout(32, 8192, 8192) == (2, 0, 128) and layout(16, 16384, 16384) == (4, 0, 128)
    assert layout(64, 16384, 16384) == (1, 0, 128)                                  # 128 clouds: no room for clusters
    assert layout(32, 2048, 4096) == (1, 0, 64)                                     # small clouds: one CTA each
    assert layout(5, 2048, 16384) == (4, 1, 28) and layout(2, 32768, 32768) == (8, 0, 32)
    assert layout(40, 2048, 16384) == (2, 1, 120) and layout(60, 2048, 16384) == (1, 0, 120)
    assert layout(32, 2048, 16384, sms=132) == (3, 1, 129) and layout(32, 2048, 16384, sms=100) == (2, 1, 96)
    for B in (1, 3, 7, 16, 31, 32, 33, 50):                                         # never more CTAs than SMs once clusters are used
        for (N, M) in ((2048, 16384), (8192, 8192), (16384, 16384), (4096, 32768)):
            cs, mixed, grid = layout(B, N, M)
            assert grid % cs == 0 and (cs == 1 or grid <= 148), (B, N, M, cs, mixed, grid)
            assert grid >= (B * cs + B if mixed else 2 * B * cs)
    with _lib.tunable(GENPC_SORT_CLUSTER="m4"):
        assert layout(32, 2048, 16384) == (4, 1, 160)
    with _lib.tunable(GENPC_SORT_CLUSTER="8"):
        assert layout(2, 700, 1300) == (8, 0, 32)
    with _lib.tunable(GENPC_SORT_CLUSTER="1"):
        assert layout(32, 2048, 16384) == (1, 0, 64)
    mixed, grid = ctypes.c_int(), ctypes.c_int()
    assert L.genpc_chamfer_sort_layout(0, 5, 5, 148, ctypes.byref(mixed), ctypes.byref(grid)) < 0
