"""Chamfer-driven 7-DoF registration (rotation 6-D + translation + log-scale) on the B200.

Mirror of the reference's optim_registration/diff_obj_pose.py for the geometric part of the loop:
ObjectPoseOptim (:339-436), get_init_rot (:470-493), build_transform (:464-468), object_pose_optimization
(:496-594).  The Pulsar point renderer and the mask losses built on it (:108-134, :286-321, :425-433) are out
of scope (BASELINE.json north_star); the loss is the reference's Chamfer term (:326-327, weight 3.0 :334).

`RegistrationBatch` is the B200-native form: any number of scans x multi-starts advance together, ONE kernel
launch per Adam iteration (csrc/register.cu), no host synchronisation until the caller reads the result.
"""
import math

import numpy as np
import torch
from torch import nn

from .. import _lib


def rotation_6d_to_matrix(d6):
    """pytorch3d.transforms.rotation_6d_to_matrix restated (rows b1, b2, b1 x b2)."""
    a1, a2 = d6[..., :3], d6[..., 3:]
    b1 = torch.nn.functional.normalize(a1, dim=-1)
    b2 = a2 - (b1 * a2).sum(-1, keepdim=True) * b1
    b2 = torch.nn.functional.normalize(b2, dim=-1)
    b3 = torch.cross(b1, b2, dim=-1)
    return torch.stack((b1, b2, b3), dim=-2)


def matrix_to_rotation_6d(matrix):
    return matrix[..., :2, :].clone().reshape(*matrix.shape[:-2], 6)


def get_init_rot(axis, angle_deg, device):
    """:470-493 -- 6-D representation of a rotation about `axis` ('x'|'y'|'z' or a 3-vector)."""
    if isinstance(axis, str):
        v = {"x": [1.0, 0.0, 0.0], "y": [0.0, 1.0, 0.0], "z": [0.0, 0.0, 1.0]}.get(axis.lower())
        if v is None:
            raise ValueError(f"unknown axis {axis}")
        axis_vec = torch.tensor(v, dtype=torch.float32)
    else:
        axis_vec = torch.as_tensor(axis, dtype=torch.float32)
        axis_vec = axis_vec / (axis_vec.norm() + 1e-8)
    a = math.radians(angle_deg)
    K = torch.tensor([[0, -axis_vec[2], axis_vec[1]], [axis_vec[2], 0, -axis_vec[0]], [-axis_vec[1], axis_vec[0], 0]])
    R = torch.eye(3) + math.sin(a) * K + (1 - math.cos(a)) * (K @ K)  # axis_angle_to_matrix (Rodrigues)
    return matrix_to_rotation_6d(R[None])[0].to(device)


def build_transform(R_obj, t, scale):
    """:464-468 -- [sR | t]; drops the c - sRc term exactly like the reference (SURVEY.md appendix B)."""
    T = torch.eye(4, device=R_obj.device)
    T[:3, :3] = R_obj * scale
    T[:3, 3] = t
    return T


class ObjectPoseOptim(nn.Module):
    """:339-436 without the renderer: same parameters (rot_6d, trans, log_scale, init scale 0.75), same buffers
    (vert_pos, center), same forward transform :419-423.  forward() returns (None, R_obj, scale[, pts]) -- the
    image slot is None because rendering is out of scope."""

    def __init__(self, vert_pos, vert_col=None, radius=None, render_size=None, device=None, R_cam=None, T_cam=None,
                 init_rot=None, focal=4.0, project_every=0):
        super().__init__()
        device = device or vert_pos.device
        self.device = device
        self.register_parameter("vert_pos", nn.Parameter(vert_pos, requires_grad=False))
        self.register_buffer("center", vert_pos.mean(0))
        if init_rot is None:
            init_rot = get_init_rot("y", 0, device)
        self.rot_6d = nn.Parameter(init_rot.clone().float())
        self.trans = nn.Parameter(torch.zeros(3, dtype=torch.float32, device=device))
        self.log_scale = nn.Parameter(torch.tensor([math.log(0.75)], dtype=torch.float32, device=device))
        self._step = 0

    def get_current_RT(self):
        R = rotation_6d_to_matrix(self.rot_6d[None])[0].detach()
        return R, self.trans.detach(), torch.exp(self.log_scale.detach())[0]

    def get_transform(self):
        R, t, s = self.get_current_RT()
        return build_transform(R, t, s)

    def forward(self, return_pts=False, project_now=False):
        self._step += 1
        R_obj = rotation_6d_to_matrix(self.rot_6d[None])[0]
        scale = torch.exp(self.log_scale)[0]
        local = (self.vert_pos - self.center) * scale
        local = (R_obj @ local.T).T
        pts = local + self.center + self.trans
        if return_pts:
            return None, R_obj, scale, pts
        return None, R_obj, scale


def pad_clouds(clouds):
    """List of [n_i,3] tensors -> (zero-padded [C, max n_i, 3] float32 tensor, lengths [C] int32), on the first cloud's device."""
    if len(clouds) == 0:
        raise ValueError("pad_clouds: no clouds")
    clouds = [torch.as_tensor(c) for c in clouds]
    for c in clouds:
        if c.dim() != 2 or c.shape[1] != 3 or c.shape[0] < 1:
            raise ValueError(f"pad_clouds: every cloud must be [n,3] with n >= 1, got {tuple(c.shape)}")
    dev = clouds[0].device
    lengths = torch.tensor([c.shape[0] for c in clouds], dtype=torch.int32)
    out = torch.zeros(len(clouds), int(lengths.max()), 3, dtype=torch.float32, device=dev)
    for i, c in enumerate(clouds):
        out[i, :c.shape[0]] = c.to(device=dev, dtype=torch.float32)
    return out, lengths.to(dev)


def cloud_centers(complete, lengths=None):
    """Centroid of every moving cloud [C,3] (register_buffer('center'), :362): over its own `lengths[i]` points when given.
    Each is the same reduction as a cloud of that size alone ([1,n,3].mean(1)), so a pair of a ragged batch and its solo
    run start from the same centre."""
    if lengths is None:
        return complete.mean(1).contiguous()
    ln = [int(v) for v in lengths.cpu()]
    return torch.stack([complete[i:i + 1, :n].mean(1)[0] for i, n in enumerate(ln)]).contiguous()


class RegistrationBatch:
    """S = C * n_starts independent pose optimisations advanced by one fused kernel launch per iteration.

    complete [C,Nc,3] (moving, e.g. generated shape), partial [C,Nr,3] (fixed scan), float32 CUDA tensors.
    Multi-start k of every cloud pair begins at Ry(k*90 deg) (:518-523), trans 0, scale 0.75 (:367-369).

    Ragged batch: complete_lengths / partial_lengths (int tensors [C], either may be omitted = full stride) give each
    pair's point counts; its points are the first rows of its stride and the rest is padding that is never read.  Each
    pair's loss is the mean over its own points and its centre the mean of its own moving points, so its trajectory is
    the one it has alone (partial sums in another order: within float rounding).  A ragged batch always runs one fused
    launch per iteration (register_step_kernel, csrc/register.cu): not the persistent kernel a small equal-size batch
    takes, nor the symmetric path that is faster above S*Nc*Nr ~ 2e8.  from_clouds() builds one from lists of clouds.
    """

    def __init__(self, complete, partial, n_starts=4, lr=0.01, w_fwd=1.0, w_inv=0.5, cd_weight=3.0, max_iters=501,
                 complete_lengths=None, partial_lengths=None):
        _lib.require_cuda(complete, partial)
        self.complete = complete.contiguous().float()
        self.partial = partial.contiguous().float()
        C, self.Nc, _ = self.complete.shape
        self.Nr = self.partial.shape[1]
        if self.partial.shape[0] != C:
            raise ValueError(f"RegistrationBatch: {C} moving clouds but {self.partial.shape[0]} fixed ones")
        dev = self.complete.device
        self.device, self.C, self.n_starts, self.S = dev, C, n_starts, C * n_starts
        self.ragged = complete_lengths is not None or partial_lengths is not None
        self.complete_lengths = self.partial_lengths = None
        if self.ragged:
            self.complete_lengths = self._lengths(complete_lengths, self.Nc, "complete_lengths")
            self.partial_lengths = self._lengths(partial_lengths, self.Nr, "partial_lengths")
        self.center = cloud_centers(self.complete, self.complete_lengths)
        p = torch.zeros(self.S, 10, device=dev)
        for k in range(n_starts):
            p[k::n_starts, :6] = get_init_rot("y", k * 90, dev)
        p[:, 9] = math.log(0.75)
        self.params = p
        self.adam_m = torch.zeros_like(p)
        self.adam_v = torch.zeros_like(p)
        self.T = max_iters
        self.loss_hist = torch.zeros(self.S, self.T, device=dev)
        self.lr, self.w_fwd, self.w_inv, self.cd_weight = lr, w_fwd, w_inv, cd_weight
        self.t = 0
        n = _lib.lib().genpc_register_workspace_bytes(self.S, self.Nc, self.Nr)
        self._ws = torch.empty(n, dtype=torch.uint8, device=dev)
        self._ws_bytes = n

    def _lengths(self, lengths, stride, name):
        """Host-side check of a per-pair point count tensor -> int32 [C] on the batch's device (None: every pair fills the stride)."""
        if lengths is None:
            return torch.full((self.C,), stride, dtype=torch.int32, device=self.device)
        ln = torch.as_tensor(lengths)
        if ln.dtype.is_floating_point or ln.dtype.is_complex or ln.dtype == torch.bool:
            raise TypeError(f"RegistrationBatch: {name} must be an integer tensor, got {ln.dtype}")
        if tuple(ln.shape) != (self.C,):
            raise ValueError(f"RegistrationBatch: {name} must have shape ({self.C},), got {tuple(ln.shape)}")
        host = ln.cpu()
        if bool((host < 1).any()) or bool((host > stride).any()):
            raise ValueError(f"RegistrationBatch: {name} must lie in [1, {stride}], got {host.tolist()}")
        return host.to(dtype=torch.int32, device=self.device).contiguous()

    @classmethod
    def from_clouds(cls, completes, partials, **kw):
        """Ragged batch from lists of [n_i,3] moving and [m_i,3] fixed clouds: zero-padded to the largest of each, with
        their point counts (pad_clouds).  Keyword arguments as for the constructor."""
        if len(completes) != len(partials):
            raise ValueError(f"from_clouds: {len(completes)} moving clouds but {len(partials)} fixed ones")
        complete, nc = pad_clouds(completes)
        partial, nr = pad_clouds(partials)
        return cls(complete, partial.to(complete.device), complete_lengths=nc, partial_lengths=nr, **kw)

    def run(self, iters):
        """Enqueue `iters` Adam iterations on the current stream (no synchronisation)."""
        if self.t + iters > self.T:
            raise _lib.GenpcError("RegistrationBatch: max_iters exceeded")
        common = (self.S, self.n_starts, self.Nc, self.Nr, int(iters), self.t, self.T, float(self.lr),
                  float(self.lr * 0.2), float(self.lr * 0.1), float(self.w_fwd), float(self.w_inv), float(self.cd_weight),
                  _lib.ptr(self._ws), self._ws_bytes, 1 if self.t == 0 else 0, _lib.current_stream(self.device))
        state = (_lib.ptr(self.params), _lib.ptr(self.adam_m), _lib.ptr(self.adam_v), _lib.ptr(self.loss_hist))
        clouds = (_lib.ptr(self.complete), _lib.ptr(self.center), _lib.ptr(self.partial))
        with torch.cuda.device(self.device):
            if self.ragged:
                rc = _lib.lib().genpc_register_run_ragged(*clouds, _lib.ptr(self.complete_lengths),
                                                          _lib.ptr(self.partial_lengths), *state, *common)
            else:
                rc = _lib.lib().genpc_register_run(*clouds, *state, *common)
        _lib.check(rc, "genpc_register_run_ragged" if self.ragged else "genpc_register_run")
        self.t += iters
        return self

    def losses(self):
        return self.loss_hist[:, :self.t]

    def best(self):
        """Per cloud pair: final params of the start with the lowest ever-seen loss (:569-576 quirk kept).
        -> (params [C,10], start index [C], best loss [C])"""
        lo = self.losses().min(1).values.view(self.C, self.n_starts)
        k = lo.argmin(1)
        sel = torch.arange(self.C, device=self.device) * self.n_starts + k
        return self.params[sel], k, lo.gather(1, k[:, None])[:, 0]

    def transforms(self):
        """4x4 [sR | t] of the best start per cloud pair (build_transform :464-468)."""
        p, _, _ = self.best()
        R = rotation_6d_to_matrix(p[:, :6])
        T = torch.eye(4, device=self.device).repeat(self.C, 1, 1)
        T[:, :3, :3] = R * torch.exp(p[:, 9])[:, None, None]
        T[:, :3, 3] = p[:, 6:9]
        return T

    def transformed(self, params=None):
        """pts = R(s(V-c))+c+t for every scan (torch ops; for inspection, not the hot path).  For a ragged batch the clouds
        keep their padded stride: rows at or past a pair's length are meaningless."""
        p = self.params if params is None else params
        per_scan = p.shape[0] == self.S
        V = self.complete.repeat_interleave(self.n_starts, 0) if per_scan else self.complete
        if self.ragged:
            c = (self.center.repeat_interleave(self.n_starts, 0) if per_scan else self.center)[:, None]
        else:
            c = V.mean(1, keepdim=True)
        R = rotation_6d_to_matrix(p[:, :6])
        local = (V - c) * torch.exp(p[:, 9])[:, None, None]
        return torch.einsum("sij,snj->sni", R, local) + c + p[:, None, 6:9]


def object_pose_optimization_points(complete_xyz, partial_xyz, lr=0.005, iters=300, cam_bias_num=4, device=None):
    """The reference's object_pose_optimization (:496-594) on in-memory clouds: 4 multi-starts x (iters+1) Adam
    steps, returns the 4x4 numpy transform of the best start."""
    device = device or torch.device("cuda:0")
    c = torch.as_tensor(complete_xyz, dtype=torch.float32, device=device)[None]
    p = torch.as_tensor(partial_xyz, dtype=torch.float32, device=device)[None]
    rb = RegistrationBatch(c, p, n_starts=cam_bias_num, lr=lr, max_iters=iters + 1)
    rb.run(iters + 1)
    return rb.transforms()[0].detach().cpu().numpy()


def object_pose_optimization_points_batch(completes, partials, lr=0.005, iters=300, cam_bias_num=4, device=None):
    """object_pose_optimization_points for many cloud pairs of any sizes in one ragged batch (lists of [n_i,3] moving and
    [m_i,3] fixed clouds): every pair runs its own 4 multi-starts x (iters+1) Adam steps, exactly as alone up to float
    rounding.  -> numpy [C,4,4], the transform of each pair's best start."""
    device = device or torch.device("cuda:0")
    cs = [torch.as_tensor(c, dtype=torch.float32, device=device) for c in completes]
    ps = [torch.as_tensor(p, dtype=torch.float32, device=device) for p in partials]
    rb = RegistrationBatch.from_clouds(cs, ps, n_starts=cam_bias_num, lr=lr, max_iters=iters + 1)
    rb.run(iters + 1)
    return rb.transforms().detach().cpu().numpy()


def load_point_cloud(point_path, device, radius=0.05, num_points=5000, seed=0):
    """:136-165 -- a .ply is read and voxel down-sampled, a .glb is surface-sampled (num_points) then down-sampled.
    -> (vert_pos [N,3], vert_col [N,3]) float32 tensors on `device`."""
    from ..utils.dataUtils import load_xyz
    from ..utils.glb import glb2point

    if str(point_path).endswith(".ply"):
        xyz, color = load_xyz(point_path, down_sample=radius)
        return torch.as_tensor(xyz, dtype=torch.float32, device=device), torch.as_tensor(color, dtype=torch.float32, device=device)
    if str(point_path).endswith(".glb"):
        return glb2point(point_path, down_sample=radius, num_points=num_points, seed=seed, device=device)
    raise ValueError("Unsupported point cloud format")


def object_pose_optimization(glb_path, point_path, radius=0.005, lr=0.005, iters=300, render_size=224, vis=False,
                             save_path=None, device=None, cam_bias_num=4):
    """Reference signature and inputs (:496-594): `point_path` = the partial scan (.ply), `glb_path` = the generated mesh
    (.glb, sampled with 120 000 points :504; a .ply is accepted too).  The Pulsar render / mask terms are out of scope:
    the loss is the Chamfer term (:326-327).  Returns the 4x4 numpy transform and saves it like the reference (:593)."""
    device = device or torch.device("cuda:0")
    partial_xyz, _ = load_point_cloud(point_path, device, radius, 8000)          # :502
    complete_xyz, _ = load_point_cloud(glb_path, device, radius, 120000)         # :504
    T = object_pose_optimization_points(complete_xyz, partial_xyz, lr, iters, cam_bias_num, device)
    np.save("final_transform.npy", T)
    return T
