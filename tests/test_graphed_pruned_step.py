"""GPU: the fused loss step captured into a CUDA graph on the pruned path.  Sort, pruned scan, fall-back and epilogue are chained
by programmatic dependent launch; inside stream capture those launches become programmatic graph edges, and the cooperative
kernel's side stream a fork / join.  The replayed step must give the eager step's outputs on changing inputs."""
import pytest
import torch

from util import shape_cloud

pytestmark = pytest.mark.gpu


def test_graphed_pruned_loss_step_equals_eager(cuda):
    from genpc_b200 import _lib
    from genpc_b200.utils.loss_util import Completionloss, GraphedLossStep

    B, N, M = 32, 2048, 16384   # BASELINE C2: the Hilbert-sorted pruned scan with the cooperative kernel on a side stream
    assert _lib.lib().genpc_chamfer_scan_kind(B, N, M) == 1
    cl = Completionloss("cd_l2")
    a0, b0 = torch.from_numpy(shape_cloud(1, B, N)).to(cuda), torch.from_numpy(shape_cloud(2, B, M)).to(cuda)
    step = GraphedLossStep(cl, a0, b0)
    for k in range(3):
        a = torch.from_numpy(shape_cloud(30 + k, B, N)).to(cuda)
        b = torch.from_numpy(shape_cloud(40 + k, B, M)).to(cuda)
        loss, ga, gb = step(a, b)
        ea = a.clone().requires_grad_(True)
        eb = b.clone().requires_grad_(True)
        el = cl.get_loss(ea, eb)
        el.backward()
        torch.cuda.synchronize()
        assert float(loss) == float(el)
        assert torch.allclose(ga, ea.grad, rtol=1e-5, atol=1e-9) and torch.allclose(gb, eb.grad, rtol=1e-5, atol=1e-9)
