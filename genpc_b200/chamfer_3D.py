"""Mirror of the reference's pybind module `chamfer_3D` (chamfer_cuda.cpp:30-33).

    forward(xyz1, xyz2, dist1, dist2, idx1, idx2) -> int
    backward(xyz1, xyz2, gradxyz1, gradxyz2, graddist1, graddist2, idx1, idx2) -> int

Same argument order, caller-allocated outputs written in place, return 1 on success (the reference
returns 1 / 0 and prints, chamfer3D.cu:145-151); failures raise instead of being silently ignored.
Work is enqueued on the CURRENT torch stream (the reference uses the legacy default stream).

Ragged batches (forward_ragged, no reference counterpart): pair b has len1[b] points at the start of its N-stride in xyz1 and
len2[b] at the start of its M-stride in xyz2 (genpc_chamfer_forward_ragged); rows past a length are never read and get
dist 0 / idx -1.  `lengths` checks such an argument.
"""
import torch

from . import _lib


def _chk(t, dtype, name):
    if t.dtype != dtype or not t.is_contiguous():
        raise _lib.GenpcError(f"{name} must be a contiguous {dtype} tensor")


def lengths(xyz1, xyz2, len1=None, len2=None):
    """Per-pair point counts of a ragged batch -> (len1, len2) as contiguous int32 [B] tensors on the clouds' device, or None
    when both are None (an equal-size batch).  An omitted side means every cloud of it fills its stride.  Shape, device and
    dtype are checked here; the values are clamped to [0, stride] on the device (no host synchronisation)."""
    if len1 is None and len2 is None:
        return None
    B = xyz1.shape[0]
    return cloud_lengths(xyz1, len1, B, "len1"), cloud_lengths(xyz2, len2, B, "len2")


def cloud_lengths(xyz, ln, B, name):
    """One side of `lengths`: the point counts `ln` of the B clouds of xyz [B,stride,3] -> contiguous int32 [B] on xyz's device
    (None: every cloud fills its stride).  Raises GenpcError for a non-tensor, a non-integer dtype, a shape other than (B,) or
    another device."""
    if ln is None:
        return torch.full((B,), xyz.shape[1], dtype=torch.int32, device=xyz.device)
    if not isinstance(ln, torch.Tensor):
        raise _lib.GenpcError(f"{name} must be a tensor")
    if ln.dtype.is_floating_point or ln.dtype.is_complex or ln.dtype == torch.bool:
        raise _lib.GenpcError(f"{name} must be an integer tensor, got {ln.dtype}")
    if tuple(ln.shape) != (B,):
        raise _lib.GenpcError(f"{name} must have shape ({B},), got {tuple(ln.shape)}")
    if ln.device != xyz.device:
        raise _lib.GenpcError(f"{name} is on {ln.device}, the clouds on {xyz.device}")
    return ln.to(torch.int32).contiguous()


def forward(xyz1, xyz2, dist1, dist2, idx1, idx2):
    return forward_ragged(xyz1, xyz2, dist1, dist2, idx1, idx2)


def forward_ragged(xyz1, xyz2, dist1, dist2, idx1, idx2, len1=None, len2=None):
    """`forward` for a ragged batch (len1 / len2: see `lengths`; both None: exactly `forward`).  A separate name keeps
    `forward`'s parameters the reference's."""
    _lib.require_cuda(xyz1, xyz2, dist1, dist2, idx1, idx2)
    for t, n in ((xyz1, "xyz1"), (xyz2, "xyz2"), (dist1, "dist1"), (dist2, "dist2")):
        _chk(t, torch.float32, n)
    for t, n in ((idx1, "idx1"), (idx2, "idx2")):
        _chk(t, torch.int32, n)
    B, N, _ = xyz1.shape
    M = xyz2.shape[1]
    lens = lengths(xyz1, xyz2, len1, len2)
    L = _lib.lib()
    with torch.cuda.device(xyz1.device):
        nbytes = L.genpc_chamfer_workspace_bytes(B, N, M)
        ws = torch.empty(max(nbytes, 8), dtype=torch.uint8, device=xyz1.device)
        stream = _lib.current_stream(xyz1.device)
        if lens is None:
            rc = L.genpc_chamfer_forward(_lib.ptr(xyz1), _lib.ptr(xyz2), _lib.ptr(dist1), _lib.ptr(dist2),
                                         _lib.ptr(idx1), _lib.ptr(idx2), B, N, M, _lib.ptr(ws), nbytes, stream)
        else:
            rc = L.genpc_chamfer_forward_ragged(_lib.ptr(xyz1), _lib.ptr(xyz2), _lib.ptr(lens[0]), _lib.ptr(lens[1]),
                                                _lib.ptr(dist1), _lib.ptr(dist2), _lib.ptr(idx1), _lib.ptr(idx2), B, N, M,
                                                _lib.ptr(ws), nbytes, None, stream)
    _lib.check(rc, "genpc_chamfer_forward" if lens is None else "genpc_chamfer_forward_ragged")
    return 1


class _StepWorkspace:
    """Scratch of one forward shape on one (device, stream): the packed-word workspace, which every successful fused call
    leaves re-armed (all-ones) so that the next call skips the memset, and the loss partials + tickets (zeroed once).  The
    cache below drops an entry when it is full or when a knob changes the size; a CUDA graph captured on an entry bakes its
    pointers in, so the graph's owner keeps a reference (GraphedLossStep.workspace)."""

    def __init__(self, device, B, N, M):
        L = _lib.lib()
        self.packed_bytes = L.genpc_chamfer_workspace_bytes(B, N, M)
        self.packed = torch.empty(max(self.packed_bytes, 8), dtype=torch.uint8, device=device)
        self.loss = torch.zeros(max(L.genpc_chamfer_fuse_workspace_bytes(B, N, M), 8), dtype=torch.uint8, device=device)
        self.armed = False


_step_ws = {}


def _step_key(device, B, N, M):
    return (device.index, torch.cuda.current_stream(device).cuda_stream, B, N, M)


def cached_step_workspace(device, B, N, M):
    """The cached workspace of this shape on the current stream of `device`, or None (nothing is created)."""
    return _step_ws.get(_step_key(device, B, N, M))


def step_workspace(device, B, N, M):
    key = _step_key(device, B, N, M)
    ws = _step_ws.get(key)
    if ws is not None and ws.packed_bytes != _lib.lib().genpc_chamfer_workspace_bytes(B, N, M):
        ws = None   # the size depends on the scan the library would pick now (a knob was flipped): start over, unarmed
        _step_ws.pop(key)
    if ws is None:
        if len(_step_ws) >= 16:   # a few live shapes at most: drop the oldest
            _step_ws.pop(next(iter(_step_ws)))
        ws = _step_ws[key] = _StepWorkspace(device, B, N, M)
    return ws


def forward_fused(xyz1, xyz2, dist1, dist2, idx1, idx2, zero1=None, zero2=None, loss=None, h_xyz1=None, h_xyz2=None,
                  chunks=6, lengths=None):
    """No pybind counterpart: `forward` through genpc_chamfer_forward_fused on a cached, re-armed workspace (no memset
    after the first call of a shape).  Whether the packed words are armed is the library's rule, not the caller's guess:
    after a successful fused call they are, on every path it may take.  zero1 / zero2: optional tensors the epilogue zero-fills (the gradient
    accumulators `backward` adds into); loss = (out_scalar, use_sqrt, w1, w2): optional fused loss reduction;
    h_xyz1 / h_xyz2: host-fed form (see forward_host); lengths = (len1, len2) as returned by `lengths()`: ragged batch
    (genpc_chamfer_forward_ragged, per-pair means in the loss), sharing the cached workspace with equal-size calls."""
    _lib.require_cuda(xyz1, xyz2, dist1, dist2, idx1, idx2)
    for t, n in ((xyz1, "xyz1"), (xyz2, "xyz2"), (dist1, "dist1"), (dist2, "dist2")):
        _chk(t, torch.float32, n)
    for t, n in ((idx1, "idx1"), (idx2, "idx2")):
        _chk(t, torch.int32, n)
    B, N, _ = xyz1.shape
    M = xyz2.shape[1]
    dev = xyz1.device
    L = _lib.lib()
    with torch.cuda.device(dev):
        ws = step_workspace(dev, B, N, M)
        out, use_sqrt, w1, w2 = loss if loss is not None else (None, 0, 0.0, 0.0)
        fuse = _lib.ChamferFuse(int(ws.armed), int(use_sqrt), float(w1), float(w2), out.data_ptr() if out is not None else None,
                                ws.loss.data_ptr(), ws.loss.numel(), zero1.data_ptr() if zero1 is not None else None,
                                zero2.data_ptr() if zero2 is not None else None)
        ws.armed = False   # stays False if the call below fails half-way
        stream = _lib.current_stream(dev)
        if lengths is not None:
            if h_xyz1 is not None:
                raise _lib.GenpcError("ragged batches have no host-fed form")
            rc = L.genpc_chamfer_forward_ragged(_lib.ptr(xyz1), _lib.ptr(xyz2), _lib.ptr(lengths[0]), _lib.ptr(lengths[1]),
                                                _lib.ptr(dist1), _lib.ptr(dist2), _lib.ptr(idx1), _lib.ptr(idx2), B, N, M,
                                                _lib.ptr(ws.packed), ws.packed_bytes, fuse, stream)
            _lib.check(rc, "genpc_chamfer_forward_ragged")
        elif h_xyz1 is None:
            rc = L.genpc_chamfer_forward_fused(_lib.ptr(xyz1), _lib.ptr(xyz2), _lib.ptr(dist1), _lib.ptr(dist2), _lib.ptr(idx1),
                                               _lib.ptr(idx2), B, N, M, _lib.ptr(ws.packed), ws.packed_bytes, fuse, stream)
            _lib.check(rc, "genpc_chamfer_forward_fused")
        else:
            if h_xyz1.is_cuda or h_xyz2.is_cuda or h_xyz1.shape != xyz1.shape or h_xyz2.shape != xyz2.shape:
                raise _lib.GenpcError("host-fed forward takes CPU clouds shaped like the device buffers")
            _chk(h_xyz1, torch.float32, "h_xyz1"), _chk(h_xyz2, torch.float32, "h_xyz2")
            rc = L.genpc_chamfer_forward_host_fused(_feed(dev), _lib.ptr(h_xyz1), _lib.ptr(h_xyz2), _lib.ptr(xyz1),
                                                    _lib.ptr(xyz2), _lib.ptr(dist1), _lib.ptr(dist2), _lib.ptr(idx1),
                                                    _lib.ptr(idx2), B, N, M, int(chunks), _lib.ptr(ws.packed), ws.packed_bytes,
                                                    fuse, stream)
            _lib.check(rc, "genpc_chamfer_forward_host_fused")
        # every fused call that reaches the scan leaves the packed words all-ones, whichever path the library took (symmetric,
        # pruned, per-direction, host-fed, ragged); an empty cloud leaves them untouched
        ws.armed = min(N, M) > 0
    return 1


_feeds = {}


def _feed(device):
    """One host-feed handle (copy stream + gate words) per device, created on first use."""
    import ctypes

    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _feeds:
        h = ctypes.c_void_p()
        with torch.cuda.device(idx):
            _lib.check(_lib.lib().genpc_host_feed_create(ctypes.byref(h)), "genpc_host_feed_create")
        _feeds[idx] = h
    return _feeds[idx]


def forward_host(h_xyz1, h_xyz2, xyz1, xyz2, dist1, dist2, idx1, idx2, chunks=6):
    """No pybind counterpart: `forward` fed from HOST tensors.  h_xyz1 / h_xyz2 (CPU, float32, contiguous; pinned for an
    asynchronous copy) are streamed into the caller-allocated CUDA tensors xyz1 / xyz2 chunk by chunk while the scan
    already consumes the chunks that have arrived (genpc_chamfer_forward_host).  Outputs as `forward`."""
    _lib.require_cuda(xyz1, xyz2, dist1, dist2, idx1, idx2)
    if h_xyz1.is_cuda or h_xyz2.is_cuda:
        raise _lib.GenpcError("forward_host takes CPU tensors as h_xyz1 / h_xyz2")
    for t, n in ((h_xyz1, "h_xyz1"), (h_xyz2, "h_xyz2"), (xyz1, "xyz1"), (xyz2, "xyz2"), (dist1, "dist1"), (dist2, "dist2")):
        _chk(t, torch.float32, n)
    for t, n in ((idx1, "idx1"), (idx2, "idx2")):
        _chk(t, torch.int32, n)
    if h_xyz1.shape != xyz1.shape or h_xyz2.shape != xyz2.shape:
        raise _lib.GenpcError("host and device clouds must have the same shape")
    B, N, _ = xyz1.shape
    M = xyz2.shape[1]
    L = _lib.lib()
    with torch.cuda.device(xyz1.device):
        nbytes = L.genpc_chamfer_workspace_bytes(B, N, M)
        ws = torch.empty(max(nbytes, 8), dtype=torch.uint8, device=xyz1.device)
        rc = L.genpc_chamfer_forward_host(_feed(xyz1.device), _lib.ptr(h_xyz1), _lib.ptr(h_xyz2), _lib.ptr(xyz1),
                                          _lib.ptr(xyz2), _lib.ptr(dist1), _lib.ptr(dist2), _lib.ptr(idx1), _lib.ptr(idx2),
                                          B, N, M, int(chunks), _lib.ptr(ws), nbytes, _lib.current_stream(xyz1.device))
    _lib.check(rc, "genpc_chamfer_forward_host")
    return 1


def host_feed_error(device):
    """True if a host-fed launch on `device` ever gave up waiting for its data (synchronises the current stream)."""
    rc = _lib.lib().genpc_host_feed_error(_feed(device), _lib.current_stream(device))
    if rc not in (0, 1):
        _lib.check(rc, "genpc_host_feed_error")
    return bool(rc)


def backward(xyz1, xyz2, gradxyz1, gradxyz2, graddist1, graddist2, idx1, idx2):
    _lib.require_cuda(xyz1, xyz2, gradxyz1, gradxyz2, graddist1, graddist2, idx1, idx2)
    for t, n in ((xyz1, "xyz1"), (xyz2, "xyz2"), (gradxyz1, "gradxyz1"), (gradxyz2, "gradxyz2"),
                 (graddist1, "graddist1"), (graddist2, "graddist2")):
        _chk(t, torch.float32, n)
    for t, n in ((idx1, "idx1"), (idx2, "idx2")):
        _chk(t, torch.int32, n)
    B, N, _ = xyz1.shape
    M = xyz2.shape[1]
    with torch.cuda.device(xyz1.device):
        rc = _lib.lib().genpc_chamfer_backward(_lib.ptr(xyz1), _lib.ptr(xyz2), _lib.ptr(graddist1),
                                               _lib.ptr(graddist2), _lib.ptr(idx1), _lib.ptr(idx2),
                                               _lib.ptr(gradxyz1), _lib.ptr(gradxyz2), B, N, M,
                                               _lib.current_stream(xyz1.device))
    _lib.check(rc, "genpc_chamfer_backward")
    return 1
