"""Chamfer distance module -- drop-in for the reference's loss_functions/Chamfer3D/dist_chamfer_3D.py (:26-74).

    dist1, dist2, idx1, idx2 = chamfer_3DDist()(input1, input2)        # [B,N,3], [B,M,3] CUDA tensors
    dist1, dist2, idx1, idx2 = chamfer_3DDist()(input1, input2, lengths1, lengths2)   # ragged batch

dist1[b,j] = min_k |input1[b,j] - input2[b,k]|^2 with idx1 the arg-min (lowest index on ties), dist2/idx2 the other
direction; differentiable w.r.t. both inputs.  GPU tensors only, exactly like the reference (:25) -- a CPU tensor
raises instead of silently falling back.

What differs from the reference is only where memory lives: outputs and gradients are created on the inputs' device
(the reference allocates them on the CPU and copies them over on every call, :33-42 and :56-60), the kernels write
every output element so no zero-fill is needed, and launches go to the current stream.

Ragged batch (no reference counterpart): lengths1 / lengths2, integer tensors [B] on the inputs' device (either may be
omitted = full stride), give each pair's point counts; pair b's points are the first rows of its stride and the rest is
padding that is never read.  Valid rows are what the pair alone gives, bit for bit; rows with no neighbour (padding, or a
pair whose other cloud is empty) get dist 0 and idx -1 and receive no gradient.  Lists of clouds: pad them with
genpc_b200.optim_registration.diff_obj_pose.pad_clouds, which returns the padded batch and its lengths.
"""
import torch
from torch import nn
from torch.autograd import Function

from ... import chamfer_3D


def _outputs(like, count):
    shape = (like.shape[0], count)
    return (torch.empty(shape, dtype=torch.float32, device=like.device),
            torch.empty(shape, dtype=torch.int32, device=like.device))


def _grad_buffers(ctx, xyz1, xyz2):
    """Gradient accumulators for a forward whose inputs need gradients: allocated now, zero-filled by the forward's
    epilogue launch (the reference zero-fills them with two launches in backward, :56-57)."""
    if any(ctx.needs_input_grad[:2]) and xyz1.dtype == torch.float32 and xyz2.dtype == torch.float32:
        return torch.empty_like(xyz1), torch.empty_like(xyz2)
    return None, None


class chamfer_3DFunction(Function):
    @staticmethod
    def forward(ctx, xyz1, xyz2, len1=None, len2=None):
        dist1, idx1 = _outputs(xyz1, xyz1.shape[1])
        dist2, idx2 = _outputs(xyz2, xyz2.shape[1])
        ctx.grads = _grad_buffers(ctx, xyz1, xyz2)
        lengths = None if len1 is None else (len1, len2)
        chamfer_3D.forward_fused(xyz1, xyz2, dist1, dist2, idx1, idx2, ctx.grads[0], ctx.grads[1], lengths=lengths)
        ctx.save_for_backward(xyz1, xyz2, idx1, idx2)
        ctx.mark_non_differentiable(idx1, idx2)
        return dist1, dist2, idx1, idx2

    @staticmethod
    def backward(ctx, graddist1, graddist2, gradidx1, gradidx2):
        xyz1, xyz2, idx1, idx2 = ctx.saved_tensors
        # the native backward ACCUMULATES (atomics), so the gradients start from zero as in the reference (:56-57):
        # the buffers zero-filled by the forward's epilogue, or fresh zeros for a second backward through the graph
        grads = ctx.grads
        ctx.grads = (None, None)
        if grads[0] is None:
            grads = torch.zeros_like(xyz1), torch.zeros_like(xyz2)
        chamfer_3D.backward(xyz1, xyz2, grads[0], grads[1], graddist1.contiguous(), graddist2.contiguous(), idx1, idx2)
        return grads + (None, None)


class chamfer_3DHostFunction(Function):
    """chamfer_3DFunction whose inputs start on the host: xyz1 / xyz2 are uninitialised CUDA leaves that the call fills
    from the CPU tensors h1 / h2 while the scan is already running on the chunks that have arrived."""

    @staticmethod
    def forward(ctx, xyz1, xyz2, h1, h2, chunks):
        dist1, idx1 = _outputs(xyz1, xyz1.shape[1])
        dist2, idx2 = _outputs(xyz2, xyz2.shape[1])
        ctx.grads = _grad_buffers(ctx, xyz1, xyz2)
        chamfer_3D.forward_fused(xyz1, xyz2, dist1, dist2, idx1, idx2, ctx.grads[0], ctx.grads[1], None, h1, h2, chunks)
        ctx.save_for_backward(xyz1, xyz2, idx1, idx2)
        ctx.mark_non_differentiable(idx1, idx2)
        return dist1, dist2, idx1, idx2

    @staticmethod
    def backward(ctx, graddist1, graddist2, gradidx1, gradidx2):
        return chamfer_3DFunction.backward(ctx, graddist1, graddist2, gradidx1, gradidx2)[:2] + (None, None, None)


def host_leaves(h1, h2, device=None):
    """Uninitialised CUDA leaf tensors shaped like the CPU clouds h1 / h2 (they receive the data and the gradients)."""
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    return (torch.empty(h1.shape, dtype=torch.float32, device=device).requires_grad_(True),
            torch.empty(h2.shape, dtype=torch.float32, device=device).requires_grad_(True))


class chamfer_3DDist(nn.Module):
    def forward(self, input1, input2, lengths1=None, lengths2=None):
        a, b = input1.contiguous(), input2.contiguous()
        lens = chamfer_3D.lengths(a, b, lengths1, lengths2)
        return chamfer_3DFunction.apply(a, b, *(lens if lens is not None else (None, None)))

    def forward_from_host(self, input1, input2, device=None, chunks=6):
        """`forward` for CPU (pinned) inputs -- the reference's `chamfer(x.cuda(), y.cuda())` with the host-to-device
        copy overlapped with the scan.  Returns (dist1, dist2, idx1, idx2, xyz1, xyz2): xyz1 / xyz2 are the CUDA copies
        of the inputs, leaves of the autograd graph (their .grad receives d/d input1, d/d input2)."""
        xyz1, xyz2 = host_leaves(input1, input2, device)
        out = chamfer_3DHostFunction.apply(xyz1, xyz2, input1.contiguous().float(), input2.contiguous().float(), chunks)
        return out + (xyz1, xyz2)
