"""Completion losses on the B200 kernels: the drop-in for the reference's `Completionloss` (utils/loss_util.py:8-53).

Same constructor argument (`'cd_l1' | 'cd_l2' | 'emd'`), same public methods and reductions:

    chamfer_l1          (mean sqrt d1 + mean sqrt d2) / 2          reference :25-29
    chamfer_l2           mean d1 + mean d2                          :31-33
    chamfer_partial_l1   mean sqrt d1                               :35-38
    chamfer_partial_l2   mean d1                                    :40-43
    emd_loss             mean_b mean_n sqrt(dist), eps .005, 50 it  :45-49
    get_loss             the metric selected by `loss_func`         :51-53

The reference wraps emdModule in nn.DataParallel (:12), i.e. one process scattering the batch over its visible
GPUs; this build's multi-GPU model is one process per GPU (genpc_b200.sharded), so the module is called directly.

Ragged batches (no reference counterpart): every Chamfer form and get_loss take gen_lengths / gt_lengths, integer tensors
[B] on the clouds' device (either may be omitted = full stride).  Each mean then runs over a pair's own points and the pairs
are averaged: (1/B) sum_b [w1 mean_{j<len1[b]} f(d1) + w2 mean_{k<len2[b]} f(d2)], a side with no points contributing 0
(genpc_chamfer_forward_ragged); with every length at its stride it is the equal-size loss.  EMD takes no lengths.
"""
import torch
from torch.autograd import Function

from .. import _lib, chamfer_3D
from ..loss_functions import chamfer_3DDist, emdModule

_EMD_EPS, _EMD_ITERS = 0.005, 50
_KNOWN = ("cd_l1", "cd_l2", "emd")


def _l1(d):
    return torch.sqrt(d).mean()


def _pair_mean(d, lengths, f):
    """(1/B) sum_b mean_{j < lengths[b]} f(d[b, j]) as literal masked torch expressions (0 for a pair with no points): the A/B
    reference of the fused ragged loss.  lengths None: f(d).mean()."""
    if lengths is None:
        return f(d).mean()
    ln = lengths.clamp(0, d.shape[1])
    mask = torch.arange(d.shape[1], device=d.device)[None, :] < ln[:, None]
    # padding rows go through f as 1 and are then dropped: sqrt's backward at a padding 0 would be 0 * inf = NaN
    s = torch.where(mask, f(torch.where(mask, d, torch.ones_like(d))), torch.zeros_like(d)).sum(1)
    return torch.where(ln > 0, s / ln.clamp(min=1), torch.zeros_like(s)).mean()


class _FusedChamferLoss(Function):
    """w1 * mean f(d1) + w2 * mean f(d2) in two launches forward (scan, epilogue: fix-up + unpack + loss reduction +
    zero-fill of the gradient accumulators + re-arming of the workspace -- genpc_chamfer_forward_fused) and one backward,
    instead of the scan plus ~16 elementwise / reduction launches of the torch expression.  Same value up to summation
    order."""

    @staticmethod
    def forward(ctx, xyz1, xyz2, use_sqrt, w1, w2, h1=None, h2=None, chunks=6, len1=None, len2=None):
        _lib.require_cuda(xyz1, xyz2)
        a, b = xyz1.contiguous().float(), xyz2.contiguous().float()
        lengths = chamfer_3D.lengths(a, b, len1, len2)
        B, N, _ = a.shape
        M = b.shape[1]
        dev = a.device
        d1 = torch.empty(B, N, device=dev)
        d2 = torch.empty(B, M, device=dev)
        i1 = torch.empty(B, N, dtype=torch.int32, device=dev)
        i2 = torch.empty(B, M, dtype=torch.int32, device=dev)
        out = torch.empty((), device=dev)
        need_grad = any(ctx.needs_input_grad[:2])
        ga = torch.empty_like(a) if need_grad else None   # zero-filled by the epilogue
        gb = torch.empty_like(b) if need_grad else None
        # host-fed when h1 / h2 are given: xyz1 / xyz2 are uninitialised leaves, filled from h1 / h2 while the scan runs
        chamfer_3D.forward_fused(a, b, d1, d2, i1, i2, ga, gb, (out, use_sqrt, w1, w2), h1, h2, chunks, lengths)
        ctx.save_for_backward(a, b, d1, d2, i1, i2)
        ctx.lengths = lengths
        ctx.cfg = (int(use_sqrt), float(w1), float(w2))
        ctx.grads = (ga, gb)
        return out

    @staticmethod
    def backward(ctx, upstream):
        a, b, d1, d2, i1, i2 = ctx.saved_tensors
        use_sqrt, w1, w2 = ctx.cfg
        B, N, _ = a.shape
        M = b.shape[1]
        ga, gb = ctx.grads
        ctx.grads = (None, None)   # a second backward through the same graph gets fresh accumulators
        if ga is None:
            ga, gb = torch.zeros_like(a), torch.zeros_like(b)
        up = upstream.contiguous().float()
        stream, ln = _lib.current_stream(a.device), ctx.lengths
        with torch.cuda.device(a.device):
            if ln is None:
                rc = _lib.lib().genpc_chamfer_loss_backward(_lib.ptr(a), _lib.ptr(b), _lib.ptr(d1), _lib.ptr(d2), _lib.ptr(i1),
                                                            _lib.ptr(i2), _lib.ptr(up), use_sqrt, w1, w2, _lib.ptr(ga),
                                                            _lib.ptr(gb), B, N, M, stream)
            else:
                rc = _lib.lib().genpc_chamfer_loss_backward_ragged(
                    _lib.ptr(a), _lib.ptr(b), _lib.ptr(ln[0]), _lib.ptr(ln[1]), _lib.ptr(d1), _lib.ptr(d2), _lib.ptr(i1),
                    _lib.ptr(i2), _lib.ptr(up), use_sqrt, w1, w2, _lib.ptr(ga), _lib.ptr(gb), B, N, M, stream)
        _lib.check(rc, "genpc_chamfer_loss_backward" if ln is None else "genpc_chamfer_loss_backward_ragged")
        return ga, gb, None, None, None, None, None, None, None, None


def _ident(d):
    return d


def _or_full(lengths, d):
    """A side's lengths as a tensor on d's device (None: every cloud fills its stride)."""
    if lengths is None:
        return torch.full((d.shape[0],), d.shape[1], dtype=torch.int64, device=d.device)
    return lengths.to(device=d.device, dtype=torch.int64)


class Completionloss:
    def __init__(self, loss_func="cd_l1"):
        if loss_func not in _KNOWN:
            raise Exception("loss function {} not supported yet!".format(loss_func))
        self.loss_func = loss_func
        self.chamfer_dist = chamfer_3DDist()
        self.EMD = emdModule()
        self.metric = {"cd_l1": self.chamfer_l1, "cd_l2": self.chamfer_l2, "emd": self.emd_loss}[loss_func]
        if loss_func != "emd":
            self.partial_matching = self.chamfer_partial_l1 if loss_func == "cd_l1" else self.chamfer_partial_l2

    # one extension call serves both directions; partial variants keep only the first cloud's distances
    def _nn(self, first, second, len1=None, len2=None):
        dist_first, dist_second, _, _ = self.chamfer_dist(first, second, len1, len2)
        return dist_first, dist_second

    # the four Chamfer reductions run fused (scan + one reduction launch; one gradient launch in backward);
    # `fused=False` keeps the literal torch expressions of the reference for A/B checks (masked per-pair means for ragged
    # batches)
    fused = True

    def _fused(self, p1, p2, use_sqrt, w1, w2, len1, len2):
        return _FusedChamferLoss.apply(p1, p2, use_sqrt, w1, w2, None, None, 6, len1, len2)

    def chamfer_l1(self, p1, p2, len1=None, len2=None):
        if self.fused:
            return self._fused(p1, p2, True, 0.5, 0.5, len1, len2)
        a, b = self._nn(p1, p2, len1, len2)
        if len1 is None and len2 is None:
            return (_l1(a) + _l1(b)) / 2
        return (_pair_mean(a, _or_full(len1, a), torch.sqrt) + _pair_mean(b, _or_full(len2, b), torch.sqrt)) / 2

    def chamfer_l2(self, p1, p2, len1=None, len2=None):
        if self.fused:
            return self._fused(p1, p2, False, 1.0, 1.0, len1, len2)
        a, b = self._nn(p1, p2, len1, len2)
        if len1 is None and len2 is None:
            return a.mean() + b.mean()
        return _pair_mean(a, _or_full(len1, a), _ident) + _pair_mean(b, _or_full(len2, b), _ident)

    def chamfer_partial_l1(self, pcd1, pcd2, len1=None, len2=None):
        if self.fused:
            return self._fused(pcd1, pcd2, True, 1.0, 0.0, len1, len2)
        a = self._nn(pcd1, pcd2, len1, len2)[0]
        return _l1(a) if len1 is None and len2 is None else _pair_mean(a, _or_full(len1, a), torch.sqrt)

    def chamfer_partial_l2(self, pcd1, pcd2, len1=None, len2=None):
        if self.fused:
            return self._fused(pcd1, pcd2, False, 1.0, 0.0, len1, len2)
        a = self._nn(pcd1, pcd2, len1, len2)[0]
        return a.mean() if len1 is None and len2 is None else _pair_mean(a, _or_full(len1, a), _ident)

    def emd_loss(self, p1, p2, len1=None, len2=None):
        if len1 is not None or len2 is not None:
            raise ValueError("emd takes no lengths: the auction needs clouds of one size n with n % 256 == 0")
        sq, _ = self.EMD(p1, p2, eps=_EMD_EPS, iters=_EMD_ITERS)
        return torch.sqrt(sq).mean(1).mean()

    def get_loss(self, gen, gt, gen_lengths=None, gt_lengths=None):
        return self.metric(gen, gt, gen_lengths, gt_lengths)

    _HOST_CFG = {"cd_l1": (True, 0.5, 0.5), "cd_l2": (False, 1.0, 1.0)}

    def get_loss_from_host(self, gen, gt, device=None, chunks=6):
        """`get_loss(gen.cuda(), gt.cuda())` for CPU (pinned) clouds, with the host-to-device copy overlapped with the
        scan (genpc_chamfer_forward_host): returns (loss, gen_cuda, gt_cuda); after `loss.backward()` the gradients are
        in gen_cuda.grad / gt_cuda.grad.  Chamfer metrics only (the EMD auction needs every point before it starts).
        If the copy never arrives (the scan gives up after ~2 s) the returned loss is NaN and
        genpc_b200.chamfer_3D.host_feed_error(device) reports and clears the condition."""
        if self.loss_func not in self._HOST_CFG:
            raise Exception("get_loss_from_host supports cd_l1 / cd_l2")
        from ..loss_functions.Chamfer3D.dist_chamfer_3D import host_leaves

        a, b = host_leaves(gen, gt, device)
        use_sqrt, w1, w2 = self._HOST_CFG[self.loss_func]
        loss = _FusedChamferLoss.apply(a, b, use_sqrt, w1, w2, gen.contiguous().float(), gt.contiguous().float(), chunks)
        return loss, a, b


class GraphedLossStep:
    """One loss step -- `loss = Completionloss(...).get_loss(gen, gt); loss.backward()` -- at a fixed shape, captured ONCE into a
    CUDA graph and replayed: the three kernels of the fused step (scan, fused epilogue, gradient) become one graph launch,
    no Python / autograd / allocator work per step.  (The reference's loop pays two extension calls, ~20 elementwise torch
    launches and six CPU allocations per step, dist_chamfer_3D.py:33-60, loss_util.py:25-43.)

        step = GraphedLossStep(Completionloss('cd_l2'), gen, gt)      # gen / gt: example CUDA tensors (shape, device)
        loss, ggen, ggt = step(gen_new, gt_new)                       # copies the inputs in, replays, returns static outputs

    `loss`, `ggen`, `ggt` are the SAME tensors on every call (overwritten by the next replay).  Passing no arguments replays on
    the current contents of `step.gen` / `step.gt` (write into them in place to avoid the copy).

    The graph owns the Chamfer workspace it was captured on (`step.workspace`, the cached scratch of this shape on
    `step.stream`): its pointers are baked into the graph, so the step keeps it alive after the process-wide cache drops it
    (more shapes than the cache holds, or a knob that changes the workspace size).

    Ragged batch: gen_lengths / gt_lengths (as for get_loss) are copied into device tensors `step.gen_lengths` /
    `step.gt_lengths` that the graph reads, so a replay takes new lengths as well as new clouds:
    step(gen_new, gt_new, gen_lengths_new, gt_lengths_new), or write into those tensors in place."""

    def __init__(self, loss_obj, gen, gt, warmup=3, gen_lengths=None, gt_lengths=None):
        _lib.require_cuda(gen, gt)
        self.loss_obj = loss_obj
        dev = gen.device
        self.gen = gen.detach().clone().float().contiguous().requires_grad_(True)
        self.gt = gt.detach().clone().float().contiguous().requires_grad_(True)
        lens = chamfer_3D.lengths(self.gen, self.gt, gen_lengths, gt_lengths)
        self.gen_lengths, self.gt_lengths = (None, None) if lens is None else (lens[0].clone(), lens[1].clone())
        self.stream = torch.cuda.Stream(device=dev)
        self.stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(self.stream):
            for _ in range(max(1, warmup)):      # also arms the per-(stream, shape) workspace: the captured step has no memset
                self.gen.grad = None
                self.gt.grad = None
                loss_obj.get_loss(self.gen, self.gt, self.gen_lengths, self.gt_lengths).backward()
        self.stream.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        self.gen.grad = None
        self.gt.grad = None
        with torch.cuda.graph(self.graph, stream=self.stream):
            loss = loss_obj.get_loss(self.gen, self.gt, self.gen_lengths, self.gt_lengths)
            loss.backward()
        with torch.cuda.stream(self.stream):   # (None for EMD: no Chamfer workspace)
            self.workspace = chamfer_3D.cached_step_workspace(dev, self.gen.shape[0], self.gen.shape[1], self.gt.shape[1])
        self.loss = loss.detach()
        self.grad_gen, self.grad_gt = self.gen.grad, self.gt.grad

    def __call__(self, gen=None, gt=None, gen_lengths=None, gt_lengths=None):
        if (gen_lengths is not None or gt_lengths is not None) and self.gen_lengths is None:
            raise ValueError("GraphedLossStep: lengths given to a step captured without lengths")
        if gen is not None:
            self.gen.data.copy_(gen, non_blocking=True)
        if gt is not None:
            self.gt.data.copy_(gt, non_blocking=True)
        if gen_lengths is not None or gt_lengths is not None:
            lens = chamfer_3D.lengths(self.gen, self.gt, gen_lengths, gt_lengths)   # (an omitted side: full stride)
            self.gen_lengths.copy_(lens[0], non_blocking=True)
            self.gt_lengths.copy_(lens[1], non_blocking=True)
        self.graph.replay()
        return self.loss, self.grad_gen, self.grad_gt
