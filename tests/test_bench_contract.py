"""bench.py's contract.  CPU: the cpu_baseline object (oracle port, torch.cdist and cKDTree legs on a bounded sample), the
workload constants BASELINE.json names, and the argument parser.  --dump-outputs: what it writes on the GPU, and that it
writes nothing on the CPU port."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_workload_is_baseline_config_c2():
    sys.path.insert(0, ROOT)
    import bench

    assert (bench.B, bench.N, bench.M) == (32, 2048, 16384)          # BASELINE.json configs[1]
    assert bench.FLOP_PER_PAIR == 8 and abs(bench.FP32_NOMINAL_TFLOPS - 74.4) < 0.1
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert "Chamfer fwd+bwd point-pairs/sec" in base["metric"]


def test_cpu_baseline_object():
    sys.path.insert(0, ROOT)
    import bench
    from genpc_b200.synthetic import pcn_batch

    part, comp = pcn_batch(0, 1, bench.N, bench.M)
    out = bench.cpu_baseline(part, comp, budget_b=1)
    assert out["kind"] == "port" and out["unit"] == "pairs/s" and out["value"] > 0 and out["cores"] >= 1 and out["sample"]
    for leg in ("torch_cdist", "scipy_ckdtree"):
        assert out[leg].get("value", 0) > 0, out[leg]


def test_help_and_defaults():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--dump-outputs"):
        assert flag in r.stdout
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 2 and "--steps" in r.stderr


def test_dump_outputs_on_the_cpu_port_writes_nothing_and_says_so(tmp_path):
    """--impl reference without a GPU or without the built reference extension times the CPU port: no GPU step ran, so
    --dump-outputs leaves DIR empty, reports `dumped_outputs: null` in the line and a note on stderr."""
    import torch

    import oracle

    if torch.cuda.is_available() and oracle.load_ref_ext("chamfer_3D") is not None:
        pytest.skip("the reference extension is built: --impl reference times it on the GPU")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, timeout=900, cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert "dumped_outputs" in line and line["dumped_outputs"] is None
    assert "--dump-outputs" in r.stderr and not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_dump_outputs_of_the_reported_path_match_the_oracle(cuda, tmp_path):
    """--dump-outputs: the loss and both gradients of the timed C2 step, float32, from the path whose time `value` reports
    (eager or CUDA graph, as `api_value` names it), equal to the oracle on the bench's seeded inputs (loss within 1e-6
    relative, gradients within 1e-5 of their scale)."""
    import numpy as np

    import bench
    import oracle

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-extras",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "out")],
                       capture_output=True, text=True, timeout=900, cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and sorted(line["dumped_outputs"]["files"]) == ["grad_gen.npy", "grad_gt.npy", "loss.npy"]
    assert line["dumped_outputs"]["path"] == ("graphed" if line["api_value"].startswith("GraphedLossStep") else "eager")
    got = {k: np.load(tmp_path / "out" / (k + ".npy")) for k in ("loss", "grad_gen", "grad_gt")}
    assert all(v.dtype == np.float32 for v in got.values())
    assert got["loss"].shape == () and got["grad_gen"].shape == (bench.B, bench.N, 3) and got["grad_gt"].shape == (bench.B, bench.M, 3)
    part, comp = bench.make_inputs(0)
    d1, d2, i1, i2 = oracle.chamfer_forward(part, comp)
    want = d1.astype(np.float64).mean() + d2.astype(np.float64).mean()
    assert abs(float(got["loss"]) - want) <= 1e-6 * want
    e1, e2 = oracle.chamfer_backward(part, comp, np.full(d1.shape, 1.0 / d1.size, np.float32),
                                     np.full(d2.shape, 1.0 / d2.size, np.float32), i1, i2)
    assert np.abs(got["grad_gen"] - e1).max() <= 1e-5 * np.abs(e1).max()
    assert np.abs(got["grad_gt"] - e2).max() <= 1e-5 * np.abs(e2).max()
