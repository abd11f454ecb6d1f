"""C3 registration timing alone (64 scans x 16384 pts, 1 start each): ms per Adam iteration, scan-iters/s, final loss."""
import json, os, sys
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from genpc_b200.optim_registration.diff_obj_pose import RegistrationBatch
from genpc_b200.synthetic import partial_view, rigid_perturb, superquadric
dev = torch.device("cuda:0")
S = int(os.environ.get("REG_SCANS", 64))
comp = np.stack([superquadric(s, 16384) for s in range(S)])
part = np.stack([rigid_perturb(partial_view(comp[s], s, 16384), s)[0] for s in range(S)])
tc, tp = torch.from_numpy(comp).to(dev), torch.from_numpy(part).to(dev)
iters = int(os.environ.get("REG_ITERS", 30))
rb = RegistrationBatch(tc, tp, n_starts=1, lr=0.01, max_iters=iters + 8)
rb.run(3); torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record(); rb.run(iters); e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1)
L = rb.losses()
print(json.dumps({"ms_per_iter": ms / iters,
                  "scan_iters_per_s": S * iters / (ms * 1e-3), "loss_last_sum": float(L[:, rb.t - 1].double().sum())}))
