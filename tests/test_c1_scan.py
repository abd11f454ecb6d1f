"""BASELINE config C1 on the REAL scan: the reference's data/01184.ply (71 372 points) against the 16 384-point synthetic
shape, batch 1.  The scan's float32 coordinates are committed (tests/golden/scan_01184_xyz.npz, made by
tests/golden/make_c1_fixture.py with an independent PLY parser); the reference extension's answer on a B200 is
tests/golden/c1_ref_chamfer.npz.  CPU: the product's PLY reader against the fixture (also written back in the original
file's layout), the oracle against the golden.  GPU: the kernels against both."""
import hashlib
import os

import numpy as np
import pytest

import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
FIX = os.path.join(HERE, "golden", "scan_01184_xyz.npz")
GOLD = os.path.join(HERE, "golden", "c1_ref_chamfer.npz")


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def scan_and_shape():
    from genpc_b200.synthetic import superquadric

    return np.load(FIX)["xyz"], superquadric(0, 16384)


def test_fixture_is_intact():
    z = np.load(FIX)
    assert z["xyz"].shape == (71372, 3) and z["xyz"].dtype == np.float32
    assert digest(z["xyz"]) == str(z["sha256"])
    lo, hi = z["xyz"].min(0), z["xyz"].max(0)          # SURVEY.md section 8d [probe]: bbox of the scan
    assert np.allclose(lo, [-0.19, -0.39, -0.38], atol=0.01) and np.allclose(hi, [0.20, 0.30, 0.14], atol=0.01)


def test_ply_reader_on_the_reference_scan(tmp_path):
    """The reference's data/01184.ply holds the scan as binary little-endian doubles x, y, z.  That file is not part of this
    repository: the committed coordinates are written back in its layout, with a header written here (not by write_ply_xyz)."""
    from genpc_b200.utils.dataUtils import load_xyz, read_ply_xyz

    want = np.load(FIX)["xyz"]
    orig = str(tmp_path / "01184.ply")
    with open(orig, "wb") as f:
        f.write(f"ply\nformat binary_little_endian 1.0\nelement vertex {len(want)}\nproperty double x\nproperty double y\n"
                "property double z\nend_header\n".encode("ascii"))
        f.write(want.astype("<f8").tobytes())
    pts, col = read_ply_xyz(orig)
    assert pts.dtype == np.float32 and np.array_equal(pts, want)
    assert col is None                                   # the fixture scans carry no colour
    pts2, col2 = load_xyz(orig)                          # utils/dataUtils.py:174-189: colour = min-max normalised xyz
    assert np.array_equal(pts2, want) and col2.shape == want.shape
    ref_col = np.clip((want - want.min(0)) / (want.max(0) - want.min(0) + 1e-8), 0, 1)
    assert np.allclose(col2, ref_col, atol=1e-6)


def test_ply_write_read_round_trip(tmp_path):
    from genpc_b200.utils.dataUtils import read_ply_xyz, write_ply_xyz

    xyz = np.load(FIX)["xyz"][:5000]
    rgb = np.random.default_rng(0).integers(0, 256, size=(5000, 3)).astype(np.float32) / 255.0
    p = str(tmp_path / "a.ply")
    write_ply_xyz(p, xyz, rgb)
    pts, col = read_ply_xyz(p)
    assert np.array_equal(pts, xyz)                      # doubles on disk hold every float32 exactly
    assert np.array_equal(np.round(col * 255), np.round(rgb * 255))
    write_ply_xyz(p, xyz)
    pts, col = read_ply_xyz(p)
    assert np.array_equal(pts, xyz) and col is None


@pytest.mark.skipif(not os.path.exists(GOLD), reason="golden not generated yet")
def test_oracle_reproduces_the_reference_on_c1():
    scan, shape = scan_and_shape()
    g = np.load(GOLD)
    assert digest(shape) == str(g["shape_sha256"]), "the synthetic C1 shape changed: regenerate the golden"
    d1, d2, i1, i2 = oracle.chamfer_forward(scan[None], shape[None])
    assert np.array_equal(i1[0], g["idx1"].astype(np.int32)) and np.array_equal(i2[0], g["idx2"])
    assert np.array_equal(d1[0].view(np.int32), g["dist1"].view(np.int32))
    assert np.array_equal(d2[0].view(np.int32), g["dist2"].view(np.int32))
    assert digest(d1[0], d2[0], i1[0], i2[0]) == str(g["sha256"])


@pytest.mark.gpu
def test_c1_on_gpu_vs_oracle_and_golden(cuda):
    import torch

    from genpc_b200.loss_functions import chamfer_3DDist

    scan, shape = scan_and_shape()
    a = torch.from_numpy(scan[None]).to(cuda).requires_grad_(True)
    b = torch.from_numpy(shape[None]).to(cuda).requires_grad_(True)
    d1, d2, i1, i2 = chamfer_3DDist()(a, b)
    got = [t.detach().cpu().numpy() for t in (d1, d2, i1, i2)]
    exp = oracle.chamfer_forward(scan[None], shape[None])
    for g_, e_, name in zip(got, exp, ("dist1", "dist2", "idx1", "idx2")):
        assert np.array_equal(g_.view(np.int32), e_.view(np.int32)), name
    if os.path.exists(GOLD):
        g = np.load(GOLD)
        assert np.array_equal(got[2][0], g["idx1"].astype(np.int32)) and np.array_equal(got[3][0], g["idx2"])
        assert np.array_equal(got[0][0].view(np.int32), g["dist1"].view(np.int32))
        assert np.array_equal(got[1][0].view(np.int32), g["dist2"].view(np.int32))
    # CD-L1 through the facade + its gradient (the metric main.py:25-29 reports on this pair)
    (torch.sqrt(d1).mean() + torch.sqrt(d2).mean()).div(2).backward()
    g1 = (0.25 / np.sqrt(exp[0].astype(np.float64)) / exp[0].size).astype(np.float32)
    g2 = (0.25 / np.sqrt(exp[1].astype(np.float64)) / exp[1].size).astype(np.float32)
    e1, e2 = oracle.chamfer_backward(scan[None], shape[None], g1, g2, exp[2], exp[3])
    assert np.abs(a.grad.cpu().numpy() - e1).max() <= 1e-5 * np.abs(e1).max()
    assert np.abs(b.grad.cpu().numpy() - e2).max() <= 1e-5 * np.abs(e2).max()
