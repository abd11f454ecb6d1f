"""Small invocation of every kernel family, meant to run under compute-sanitizer (memcheck / racecheck)."""
import os, sys
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from genpc_b200 import depth as D
from genpc_b200.fps import furthest_point_sample
from genpc_b200.loss_functions import chamfer_3DDist, emdModule
from genpc_b200.optim_registration.diff_obj_pose import RegistrationBatch
from genpc_b200.sharded import nn_partial_packed, nn_unpack
dev = torch.device("cuda:0")
g = torch.Generator().manual_seed(0)
for (B, N, M) in [(2, 700, 1300), (1, 3000, 999), (2, 100, 37)]:   # sym path, sym with tails, scan path
    a = torch.rand(B, N, 3, generator=g).to(dev).requires_grad_(True); b = torch.rand(B, M, 3, generator=g).to(dev).requires_grad_(True)
    d1, d2, i1, i2 = chamfer_3DDist()(a, b); (d1.mean() + d2.mean()).backward()
x = torch.rand(2, 512, 3, generator=g).to(dev); y = torch.rand(2, 512, 3, generator=g).to(dev)
emdModule()(x, y, 0.005, 10)
furthest_point_sample(torch.rand(2, 5000, 3, generator=g).to(dev), 64, 0)
furthest_point_sample(torch.rand(1, 40000, 3, generator=g).to(dev), 8, 0)
pts = torch.rand(3000, 3, generator=g).to(dev) - 0.5
cams, _ = D.create_cameras(3, 1.6, 49.1, 64, dev)
ndc, uv, bnd = D.project_uv(cams, pts); r = D.zbuffer_render(uv, ndc, 64, 2); D.unproject(cams, bnd, r["zbuf"], ndc)
for (nc, nr) in [(1500, 900), (20000, 12000)]:                      # single-launch path and symmetric two-launch path
    rb = RegistrationBatch(torch.rand(1, nc, 3, generator=g).to(dev) - 0.5, torch.rand(1, nr, 3, generator=g).to(dev) - 0.5, n_starts=2)
    rb.run(2)
p = nn_partial_packed(torch.rand(1, 2000, 3, generator=g).to(dev), torch.rand(1, 700, 3, generator=g).to(dev), 100); nn_unpack(p)
# fused loss step (epilogue with loss reduction, zero-fill with odd tails, re-armed workspace), twice per shape; host-fed
from genpc_b200.utils.loss_util import Completionloss
from genpc_b200.reg_xyz import knn_mean_distance
from genpc_b200.sharded import sharded_chamfer_forward
cl = Completionloss("cd_l1")
for (B, N, M) in [(3, 701, 1303), (1, 3001, 997), (2, 100, 37)]:
    for _ in range(2):
        a = torch.rand(B, N, 3, generator=g).to(dev).requires_grad_(True); b = torch.rand(B, M, 3, generator=g).to(dev).requires_grad_(True)
        cl.get_loss(a, b).backward()
ha, hb = torch.rand(4, 600, 3, generator=g).pin_memory(), torch.rand(4, 1500, 3, generator=g).pin_memory()
loss, da, db = cl.get_loss_from_host(ha, hb, device=dev, chunks=2); loss.backward()
knn_mean_distance(torch.rand(3001, 3, generator=g).to(dev), 20, True); knn_mean_distance(torch.rand(17, 3, generator=g).to(dev), 32, False)
sharded_chamfer_forward(torch.rand(1, 5001, 3, generator=g).to(dev), torch.rand(1, 3003, 3, generator=g).to(dev))
from genpc_b200.reg_xyz import icp_point_to_point
icp_point_to_point(torch.rand(5, 333, 3, generator=g).to(dev), torch.rand(1, 777, 3, generator=g).to(dev), 0.3, max_iteration=3)
# ---- r02 kernels: mesh sampler, persistent small registration (one launch, several iterations), NaN points, graphed loss step
from genpc_b200 import _lib
from genpc_b200.synthetic import superquadric_mesh
from genpc_b200.utils.glb import sample_mesh
from genpc_b200.utils.loss_util import GraphedLossStep
v, f, col = superquadric_mesh(1, 12, 20)
sample_mesh(torch.from_numpy(v).to(dev), torch.from_numpy(f).to(dev), 3001, 5, torch.from_numpy(col).to(dev), return_face=True)
rb = RegistrationBatch(torch.rand(1, 1300, 3, generator=g).to(dev) - 0.5, torch.rand(1, 900, 3, generator=g).to(dev) - 0.5, n_starts=3)
rb.run(5)
a = torch.rand(2, 700, 3, generator=g); a[0, 3] = float("nan"); a[1, 5] = 3e38
d1, d2, i1, i2 = chamfer_3DDist()(a.to(dev).requires_grad_(True), torch.rand(2, 1300, 3, generator=g).to(dev).requires_grad_(True))
(d1[:, 10:].mean() + d2.mean()).backward()
step = GraphedLossStep(cl, torch.rand(2, 600, 3, generator=g).to(dev), torch.rand(2, 1500, 3, generator=g).to(dev))
step(); step()
# ---- r02 (late): pruned EMD Bid (both target sorts, spread tail at n = 4096), pruned Chamfer scans (one-CTA sort / grid sort
# with probe and forced), out-of-range hand-over
for n_, it_ in ((1024, 6), (4096, 3)):
    emdModule()(torch.rand(2, n_, 3, generator=g).to(dev), torch.rand(2, n_, 3, generator=g).to(dev), 0.005, it_)
with _lib.tunable(GENPC_EMD_SORT="bitonic"):
    emdModule()(torch.rand(1, 1280, 3, generator=g).to(dev), torch.rand(1, 1280, 3, generator=g).to(dev), 0.005, 4)
with _lib.tunable(GENPC_EMD_PRUNE="0"):
    emdModule()(torch.rand(1, 1024, 3, generator=g).to(dev), torch.rand(1, 1024, 3, generator=g).to(dev), 0.005, 4)
for knob in ("1", "2"):
    with _lib.tunable(GENPC_CHAMFER_PRUNE=knob):
        for (B, N, M) in [(2, 700, 1300), (1, 3000, 999), (1, 64, 513)]:
            chamfer_3DDist()(torch.rand(B, N, 3, generator=g).to(dev), torch.rand(B, M, 3, generator=g).to(dev))
        bad = torch.rand(1, 900, 3, generator=g); bad[0, 7, 1] = float("inf")
        chamfer_3DDist()(bad.to(dev), torch.rand(1, 700, 3, generator=g).to(dev))
chamfer_3DDist()(torch.rand(1, 70000, 3, generator=g).to(dev), torch.rand(1, 66000, 3, generator=g).to(dev))   # default: probe + grid scan
# pruned scan inside the registration loop (forced on a small symmetric-path problem), host-fed batch through the chunked pruned path
with _lib.tunable(GENPC_REGISTER_PRUNE="1", GENPC_REGISTER_MODE="sym"):
    rb = RegistrationBatch(torch.rand(2, 3000, 3, generator=g).to(dev) - 0.5, torch.rand(2, 2100, 3, generator=g).to(dev) - 0.5, n_starts=2)
    rb.run(2); rb.run(1)
with _lib.tunable(GENPC_HOST_PRUNE="1", GENPC_CHAMFER_PRUNE="1"):
    ha2, hb2 = torch.rand(6, 700, 3, generator=g).pin_memory(), torch.rand(6, 1500, 3, generator=g).pin_memory()
    loss, da, db = Completionloss("cd_l2").get_loss_from_host(ha2, hb2, device=dev, chunks=3); loss.backward()
# r02w: the sort kernel as thread-block clusters (sibling histograms / boxes through distributed shared memory, cross-CTA reads of the
# sorted records), every layout, ragged sizes
for layout in ("2", "3", "4", "8", "m2", "m3", "m4"):
    with _lib.tunable(GENPC_CHAMFER_PRUNE="1", GENPC_SORT_CLUSTER=layout):
        for (B, N, M) in [(3, 700, 5300), (2, 2048, 9000), (1, 64, 513)]:
            chamfer_3DDist()(torch.rand(B, N, 3, generator=g).to(dev), torch.rand(B, M, 3, generator=g).to(dev))
torch.cuda.synchronize(); print("sanitize smoke done")
