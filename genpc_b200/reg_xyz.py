"""Scale / ICP search of the Geometric-Preserving-Fusion stage on the GPU (reference: reg_xyz.py).

The reference scores 11 isotropic + 1000 anisotropic scale candidates one at a time: deepcopy -> Open3D ICP on the
CPU -> H2D -> two Chamfer extension calls (4 NN scans) -> `cd < best_loss` D2H sync (reg_xyz.py:60-96, 146-173).
Here the candidates ARE the batch dimension: one batched point-to-point ICP (NN from the Chamfer kernel + one
genpc_icp_step launch per iteration: inliers, covariance, Horn's closed-form rotation, convergence) and one Chamfer call
score all of them, everything stays on the device.

Open3D is not vendored: `registration_icp` (point-to-point, default criteria: 30 iterations, relative fitness /
RMSE 1e-6), voxel down-sampling and `remove_statistical_outlier` are restated from their documented behaviour
(parity unpinned, SURVEY.md appendix B).  Function names and argument meaning follow the reference.
"""
import os

import numpy as np
import torch

from . import _lib, chamfer_3D
from .fps import furthest_point_sample
from .loss_functions import chamfer_3DDist
from .optim_registration.diff_obj_pose import object_pose_optimization_points, pad_clouds
from .utils.dataUtils import normalize_numpy, voxel_down_sample  # noqa: F401

_cd = chamfer_3DDist()


def _apply(T, pts):
    """T [K,4,4], pts [K,N,3] -> transformed points."""
    return pts @ T[:, :3, :3].transpose(1, 2) + T[:, None, :3, 3]


def chamfer_partial_l1_batched(src, tgt, cd_inv_weight=0.0, src_lengths=None, tgt_lengths=None):
    """Per-candidate score of the reference's sweep (reg_xyz.py:81-84, 167-170):
    CDp-L1(src->tgt) + cd_inv_weight * CDp-L1(tgt->src), src [K,Ns,3], tgt [K,Nt,3] -> [K].
    src_lengths / tgt_lengths (integer tensors [K], either may be omitted = full stride): ragged batch, each candidate's
    means taken over its own points (a side with no points contributes 0)."""
    src, tgt = src.contiguous(), tgt.contiguous()
    lens = chamfer_3D.lengths(src, tgt, src_lengths, tgt_lengths)
    if lens is None:
        d1, d2, _, _ = _cd(src, tgt)
        return torch.sqrt(d1).mean(1) + cd_inv_weight * torch.sqrt(d2).mean(1)
    d1, d2, _, _ = _cd(src, tgt, *lens)   # rows past a length come back as dist 0
    n1, n2 = (ln.clamp(min=1).float() for ln in lens)
    return torch.sqrt(d1).sum(1) / n1 + cd_inv_weight * (torch.sqrt(d2).sum(1) / n2)


def _candidate_lengths(source, target, source_lengths, target_lengths):
    """Lengths of a ragged ICP batch -> int32 [K] pair, checked as chamfer_3D.lengths does; a [1] target length of a shared
    [1,Nt,3] target is expanded with it."""
    K = source.shape[0]
    if isinstance(target_lengths, torch.Tensor) and tuple(target_lengths.shape) == (1,) and target.shape[0] == 1 and K > 1:
        target_lengths = target_lengths.expand(K)
    return chamfer_3D.lengths(source, target.expand(K, -1, -1), source_lengths, target_lengths)


def icp_point_to_point(source, target, max_correspondence_distance=0.05, init_transform=None, max_iteration=30,
                       relative_fitness=1e-6, relative_rmse=1e-6, source_lengths=None, target_lengths=None):
    """Batched Open3D-style registration_icp (TransformationEstimationPointToPoint, no scaling), reg_xyz.py:9-38.
    source [K,Ns,3], target [K,Nt,3] (or [1,Nt,3]) -> (T [K,4,4], fitness [K], inlier_rmse [K]).
    Per iteration: transform (one bmm), nearest neighbours of all candidates (one Chamfer launch pair) and ONE
    genpc_icp_step launch (inliers, fitness / rmse / convergence, covariance, Horn rotation, T update) -- no host
    synchronisation except a convergence poll every 4 iterations.  GENPC_ICP_TORCH=1 selects the torch formulation
    (batched float64 SVD, ~25 launches and a host sync per iteration) the kernel replaced; both agree to rounding.
    source_lengths [K] / target_lengths [K] (or [1] with a shared target; integer tensors on the clouds' device, either may be
    omitted = full stride): ragged batch, candidate k has its first source_lengths[k] / target_lengths[k] points and the rest
    is padding that is never read.  Its results are bit for bit what it gets alone; see _icp_point_to_point_ragged."""
    if source_lengths is not None or target_lengths is not None:
        if os.environ.get("GENPC_ICP_TORCH") == "1":
            raise _lib.GenpcError("GENPC_ICP_TORCH=1 has no ragged form: drop the lengths or the knob")
        T, state = _icp_point_to_point_ragged(source, target, max_correspondence_distance, init_transform, max_iteration,
                                              relative_fitness, relative_rmse, source_lengths, target_lengths)
        return T, state[:, 0].clone(), state[:, 1].clone()
    if os.environ.get("GENPC_ICP_TORCH") == "1":
        return _icp_point_to_point_torch(source, target, max_correspondence_distance, init_transform, max_iteration,
                                         relative_fitness, relative_rmse)
    _lib.require_cuda(source, target)
    K, Ns, _ = source.shape
    dev = source.device
    source = source.contiguous().float()
    tgt = target.float()
    if tgt.shape[0] == 1 and K > 1:
        tgt = tgt.expand(K, -1, -1)
    tgt = tgt.contiguous()
    Nt = tgt.shape[1]
    T = torch.eye(4, device=dev).repeat(K, 1, 1) if init_transform is None else \
        torch.as_tensor(init_transform, dtype=torch.float32, device=dev).expand(K, 4, 4).clone()
    T = T.contiguous()
    state = torch.zeros(K, 4, device=dev)
    thr2 = float(max_correspondence_distance) ** 2
    L = _lib.lib()
    with torch.no_grad(), torch.cuda.device(dev):
        for it in range(max_iteration + 1):
            cur = _apply(T, source).contiguous()
            d1, _, i1, _ = _cd(cur, tgt)
            rc = L.genpc_icp_step(_lib.ptr(cur), _lib.ptr(tgt), _lib.ptr(d1), _lib.ptr(i1), _lib.ptr(T), _lib.ptr(state), K, Ns,
                                  K, Nt, thr2, float(relative_fitness), float(relative_rmse), int(it < max_iteration),
                                  _lib.current_stream(dev))
            _lib.check(rc, "genpc_icp_step")
            if it % 4 == 3 and bool(state[:, 2].all()):   # every candidate converged: the remaining iterations are no-ops
                break
    return T, state[:, 0].clone(), state[:, 1].clone()


def _icp_point_to_point_ragged(source, target, max_correspondence_distance, init_transform, max_iteration, relative_fitness,
                               relative_rmse, source_lengths, target_lengths):
    """icp_point_to_point for a ragged batch: a transform-only genpc_icp_step_ragged call writes cur = T source, then per
    iteration one ragged Chamfer call over the candidates that have not converged (scan_len) and one genpc_icp_step_ragged
    launch, which also writes the next cur.  Same convergence poll as the equal-size loop.  A candidate's arithmetic does not
    depend on its batch, so the batch runs until its slowest candidate converges and each one ends as it would alone.
    -> (T [K,4,4], state [K,4] = fitness, inlier_rmse, converged, calls)."""
    src_len, tgt_len = _candidate_lengths(source, target, source_lengths, target_lengths)
    _lib.require_cuda(source, target)
    K, Ns, _ = source.shape
    dev = source.device
    source = source.contiguous().float()
    tgt = target.float()
    if tgt.shape[0] == 1 and K > 1:
        tgt = tgt.expand(K, -1, -1)   # the ragged Chamfer takes one target per pair
    tgt = tgt.contiguous()
    Nt = tgt.shape[1]
    T = torch.eye(4, device=dev).repeat(K, 1, 1) if init_transform is None else \
        torch.as_tensor(init_transform, dtype=torch.float32, device=dev).expand(K, 4, 4).clone()
    T = T.contiguous()
    state = torch.zeros(K, 4, device=dev)
    cur = torch.zeros_like(source)
    scan_len = torch.empty(K, dtype=torch.int32, device=dev)
    thr2 = float(max_correspondence_distance) ** 2
    L = _lib.lib()

    def step(d1, i1, update):
        rc = L.genpc_icp_step_ragged(_lib.ptr(source), _lib.ptr(cur), _lib.ptr(tgt), _lib.ptr(d1), _lib.ptr(i1),
                                     _lib.ptr(src_len), _lib.ptr(tgt_len), _lib.ptr(scan_len), _lib.ptr(T), _lib.ptr(state),
                                     K, Ns, K, Nt, thr2, float(relative_fitness), float(relative_rmse), int(update),
                                     _lib.current_stream(dev))
        _lib.check(rc, "genpc_icp_step_ragged")

    with torch.no_grad(), torch.cuda.device(dev):
        step(None, None, 0)
        for it in range(max_iteration + 1):
            d1, _, i1, _ = _cd(cur, tgt, scan_len, tgt_len)
            step(d1, i1, it < max_iteration)
            if it % 4 == 3 and bool(state[:, 2].all()):
                break
    return T, state


def _icp_point_to_point_torch(source, target, max_correspondence_distance=0.05, init_transform=None, max_iteration=30,
                              relative_fitness=1e-6, relative_rmse=1e-6):
    """The torch formulation of icp_point_to_point (kept for A/B checks: tests/test_reg_xyz.py)."""
    K, Ns, _ = source.shape
    dev = source.device
    if target.shape[0] == 1 and K > 1:
        target = target.expand(K, -1, -1)
    target = target.contiguous()
    T = torch.eye(4, device=dev).repeat(K, 1, 1) if init_transform is None else \
        torch.as_tensor(init_transform, dtype=torch.float32, device=dev).expand(K, 4, 4).clone()
    thr2 = float(max_correspondence_distance) ** 2
    active = torch.ones(K, dtype=torch.bool, device=dev)
    fit_prev = torch.zeros(K, device=dev)
    rmse_prev = torch.zeros(K, device=dev)
    fitness = torch.zeros(K, device=dev)
    rmse = torch.zeros(K, device=dev)
    for it in range(max_iteration + 1):
        cur = _apply(T, source)
        d1, _, i1, _ = _cd(cur.contiguous(), target)
        inl = d1 < thr2
        cnt = inl.sum(1).clamp(min=1).float()
        fitness = inl.sum(1).float() / Ns
        rmse = torch.sqrt((d1 * inl).sum(1) / cnt)
        if it > 0:
            conv = ((fitness - fit_prev).abs() < relative_fitness) & ((rmse - rmse_prev).abs() < relative_rmse)
            active = active & ~conv
        if it == max_iteration or not bool(active.any()):
            break
        fit_prev, rmse_prev = fitness, rmse
        # Kabsch on the inlier correspondences (cur -> target[nn])
        nn = torch.gather(target, 1, i1.long()[..., None].expand(-1, -1, 3))
        w = inl.float()[..., None]
        mu_s = (cur * w).sum(1) / cnt[:, None]
        mu_t = (nn * w).sum(1) / cnt[:, None]
        H = ((cur - mu_s[:, None]) * w).transpose(1, 2) @ (nn - mu_t[:, None])
        U, _, Vh = torch.linalg.svd(H.double())
        V, Ut = Vh.transpose(1, 2), U.transpose(1, 2)
        D = torch.eye(3, dtype=torch.float64, device=dev).repeat(K, 1, 1)
        D[:, 2, 2] = torch.sign(torch.linalg.det(V @ Ut))
        R = (V @ D @ Ut).float()
        t = mu_t - (R @ mu_s[..., None])[..., 0]
        upd = torch.eye(4, device=dev).repeat(K, 1, 1)
        upd[:, :3, :3], upd[:, :3, 3] = R, t
        ok = (active & (inl.sum(1) >= 3))[:, None, None]
        T = torch.where(ok, upd @ T, T)
    return T, fitness, rmse


def icp_with_scaling_xyz(source, target, scales, max_correspondence_distance=0.05, init_transform=None):
    """reg_xyz.py:9-21 batched: scale the source per axis (scales [K,3]) then ICP.  Returns (scaled source, T, fitness, rmse)."""
    scales = torch.as_tensor(scales, dtype=torch.float32, device=source.device)
    src = source[None] * scales[:, None, :] if source.dim() == 2 else source * scales[:, None, :]
    T, f, r = icp_point_to_point(src, target if target.dim() == 3 else target[None], max_correspondence_distance,
                                 init_transform)
    return src, T, f, r


def icp_with_scaling(source, target, scale, max_correspondence_distance=0.05, init_transform=None):
    """reg_xyz.py:24-38 batched over `scale` [K]: ICP, then ICP again from result @ diag(scale)."""
    scale = torch.as_tensor(scale, dtype=torch.float32, device=source.device).reshape(-1)
    K = scale.shape[0]
    src = source[None].expand(K, -1, -1).contiguous()
    tgt = target[None].contiguous()
    T0, _, _ = icp_point_to_point(src, tgt, max_correspondence_distance, init_transform)
    S = torch.eye(4, device=source.device).repeat(K, 1, 1)
    S[:, 0, 0] = S[:, 1, 1] = S[:, 2, 2] = scale
    return icp_point_to_point(src, tgt, max_correspondence_distance, T0 @ S)


def coarse_scale_sweep(s_down, t_down, scales, max_correspondence_distance=0.075, cd_inv_weight=0.5):
    """The coarse sweep of reg() for one object (reg_xyz.py:146-173): icp_with_scaling over `scales`, then every candidate
    scored by partial CD-L1 of the scan against the target moved by the inverse transform; the first minimum wins.
    s_down [Ns,3] / t_down [Nt,3]: the voxel down-sampled scan and generated shape.
    -> {"best_scale": float, "coarse_loss": float, "coarse_transformation": [4,4] tensor}."""
    Ts, _, _ = icp_with_scaling(s_down, t_down, scales, max_correspondence_distance)
    inv = torch.linalg.inv(Ts.double()).float()
    t_moved = _apply(inv, t_down[None].expand(len(scales), -1, -1))
    cd = chamfer_partial_l1_batched(s_down[None].expand(len(scales), -1, -1), t_moved, cd_inv_weight)
    k = int(torch.argmin(cd))
    return {"best_scale": float(scales[k]), "coarse_loss": float(cd[k]), "coarse_transformation": Ts[k]}


def coarse_scale_sweep_batch(sources, targets, scales=np.linspace(1.5, 0.8, 11), max_correspondence_distance=0.075,
                             cd_inv_weight=0.5):
    """coarse_scale_sweep for a dataset of objects of different sizes in one ragged batch.  sources / targets: lists of
    [n_i,3] CUDA tensors, already down-sampled (object i = (sources[i], targets[i])).  -> one dict per object, with the keys
    of coarse_scale_sweep.

    The first ICP pass of icp_with_scaling starts from the identity whatever the scale, so it runs once per object (O
    candidates, not len(scales)·O); the second pass runs from T0 @ diag(s) over the len(scales)·O (object, scale) candidates
    (object-major).  Each object's transforms are bit for bit those it gets alone in this function; against
    coarse_scale_sweep they differ by rounding only (the ragged loop transforms the clouds with its own fma order, not a
    bmm), and the losses are per-candidate means over the object's own points."""
    if len(sources) != len(targets):
        raise ValueError(f"coarse_scale_sweep_batch: {len(sources)} sources but {len(targets)} targets")
    src, src_len = pad_clouds(sources)
    tgt, tgt_len = pad_clouds(targets)
    O, S = src.shape[0], len(scales)
    dev = src.device
    T0, _, _ = icp_point_to_point(src, tgt, max_correspondence_distance, source_lengths=src_len, target_lengths=tgt_len)
    sc = torch.as_tensor(np.asarray(scales), dtype=torch.float32, device=dev)
    D = torch.eye(4, device=dev).repeat(S, 1, 1)
    D[:, 0, 0] = D[:, 1, 1] = D[:, 2, 2] = sc
    init = T0.repeat_interleave(S, 0) @ D.repeat(O, 1, 1)
    src2, tgt2 = src.repeat_interleave(S, 0), tgt.repeat_interleave(S, 0)
    sl2, tl2 = src_len.repeat_interleave(S), tgt_len.repeat_interleave(S)
    Ts, _, _ = icp_point_to_point(src2, tgt2, max_correspondence_distance, init, source_lengths=sl2, target_lengths=tl2)
    inv = torch.linalg.inv(Ts.double()).float()
    cd = chamfer_partial_l1_batched(src2, _apply(inv, tgt2), cd_inv_weight, sl2, tl2).view(O, S)
    k = torch.argmin(cd, 1)   # first minimum per object, as coarse_scale_sweep
    loss = cd.gather(1, k[:, None])[:, 0].cpu().tolist()
    k = k.cpu().tolist()
    return [{"best_scale": float(scales[k[o]]), "coarse_loss": float(loss[o]), "coarse_transformation": Ts[o * S + k[o]]}
            for o in range(O)]


def iterative_scale_search(source_xyz, target_xyz, scale_ranges, scale_steps, init_transform=None, cd_inv_weight=0.0,
                           chunk=250):
    """reg_xyz.py:60-96: scale_steps^3 anisotropic candidates (z outer, x, y inner -- the reference's loop order, so
    `cd < best_loss` ties resolve identically: first candidate wins), each ICP-refined and scored by partial CD-L1.
    Returns (best_scales_transformation 4x4 np, best_loss float, best_transformation 4x4 np)."""
    dev = source_xyz.device
    xs = np.linspace(scale_ranges[0][0], scale_ranges[0][1], scale_steps)
    ys = np.linspace(scale_ranges[1][0], scale_ranges[1][1], scale_steps)
    zs = np.linspace(scale_ranges[2][0], scale_ranges[2][1], scale_steps)
    cand = np.array([[x, y, z] for z in zs for x in xs for y in ys], dtype=np.float32)
    losses, Ts = [], []
    for c0 in range(0, len(cand), chunk):
        sc = torch.from_numpy(cand[c0:c0 + chunk]).to(dev)
        src, T, _, _ = icp_with_scaling_xyz(source_xyz, target_xyz, sc, 0.075, init_transform)
        tgt = target_xyz[None].expand(src.shape[0], -1, -1)
        # the reference scores the SCALED (not ICP-transformed) source copy against the target (:79-84)
        losses.append(chamfer_partial_l1_batched(src, tgt, cd_inv_weight))
        Ts.append(T)
    losses, Ts = torch.cat(losses), torch.cat(Ts)
    k = int(torch.argmin(losses))  # argmin returns the first minimum == the reference's strict `<` update
    best = np.eye(4)
    best[0, 0], best[1, 1], best[2, 2] = cand[k]
    return best, float(losses[k]), Ts[k].double().cpu().numpy()


def remove_close_points(source_xyz, target_xyz, distance_threshold=0.0001):
    """reg_xyz.py:41-57: keep the target points whose nearest source point is at squared distance >= threshold
    (Open3D's KD-tree returns squared distances).  One NN launch instead of a Python loop of KD-tree queries."""
    d1, _, _, _ = _cd(target_xyz[None].contiguous(), source_xyz[None].contiguous())
    return d1[0] >= distance_threshold


def knn_mean_distance(xyz, k, include_self=True, lengths=None):
    """Mean distance from each point of xyz [N,3] (CUDA) to its k nearest points of the same cloud
    (genpc_knn_mean_distance; include_self counts the point itself, as a KD-tree query of a cloud point does).
    A batch xyz [B,N,3] -> [B,N] in one launch (genpc_knn_mean_distance_ragged): lengths (integer tensor [B] on the clouds'
    device, None = every cloud fills the stride) gives each cloud's point count, its points being the first rows of its stride.
    Each cloud's rows are bit for bit its solo call on its own points; rows past a length are never read and come back -1.
    The lengths are clamped to [0, N] on the device, so the call does not synchronise with the host."""
    if xyz.dim() == 2 and lengths is not None:
        raise _lib.GenpcError("lengths need a batch of clouds [B,N,3], got one cloud [N,3]")
    if xyz.dim() not in (2, 3) or xyz.shape[-1] != 3:
        raise _lib.GenpcError(f"knn_mean_distance takes [N,3] or [B,N,3] clouds, got {tuple(xyz.shape)}")
    if xyz.dim() == 3:
        ln = chamfer_3D.cloud_lengths(xyz, lengths, xyz.shape[0], "lengths")
    _lib.require_cuda(xyz)
    x = xyz.contiguous().float()
    out = torch.empty(x.shape[:-1], dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        if x.dim() == 2:
            rc = _lib.lib().genpc_knn_mean_distance(_lib.ptr(x), x.shape[0], int(k), int(bool(include_self)), _lib.ptr(out),
                                                    _lib.current_stream(x.device))
        else:
            rc = _lib.lib().genpc_knn_mean_distance_ragged(_lib.ptr(x), _lib.ptr(ln), x.shape[0], x.shape[1], int(k),
                                                           int(bool(include_self)), _lib.ptr(out), _lib.current_stream(x.device))
    _lib.check(rc, "genpc_knn_mean_distance" if x.dim() == 2 else "genpc_knn_mean_distance_ragged")
    return out


def statistical_outlier_mask(mean_dist, std_ratio):
    """Open3D's threshold over per-point k-NN means [..., N] (the last axis is one cloud) -> bool keep mask of the same shape:
    keep 0 < mean < cloud_mean + std_ratio * std_dev, in float64.  Only means > 0 enter the sums (a mean of exactly 0 comes from
    duplicated points); the divisors count every answered query (mean >= 0, so -1 rows -- padding, or a query that found
    nothing -- count nowhere); std_dev divides by n_valid - 1 and is 0 below two answered queries.  Masked reductions, no
    boolean indexing: no host synchronisation, and a cloud with nothing answered keeps nothing."""
    md = mean_dist.double()
    pos = md > 0
    nv = (md >= 0).sum(-1, keepdim=True)
    mu = torch.where(pos, md, 0.0).sum(-1, keepdim=True) / nv.clamp(min=1)
    ss = torch.where(pos, (md - mu) ** 2, 0.0).sum(-1, keepdim=True)
    sd = torch.where(nv > 1, torch.sqrt(ss / (nv - 1).clamp(min=1)), 0.0)
    return pos & (md < mu + std_ratio * sd)


def remove_statistical_outlier(xyz, nb_neighbors=20, std_ratio=2.5, lengths=None):
    """Open3D remove_statistical_outlier as the reference uses it (reg_xyz.py:219, utils/dataUtils.py:652-666),
    restated on the k-NN kernel: per point the mean distance to its nb_neighbors nearest points -- the KD-tree query of
    a cloud point returns the point itself first, so it is one of them -- then statistical_outlier_mask's threshold.
    xyz [N,3] -> bool keep mask [N]; a batch xyz [B,N,3] with lengths as knn_mean_distance -> [B,N], every cloud thresholded
    over its own points and padding rows False.  No host synchronisation in either form.  (Open3D is not vendored: semantics
    from its documented behaviour, parity unpinned; the oracle defines them.)"""
    return statistical_outlier_mask(knn_mean_distance(xyz, nb_neighbors, True, lengths), std_ratio)


def get_rotate_matrix(axis, angle):
    """utils/dataUtils.py:455-471 (degrees)."""
    a = angle * np.pi / 180
    c, s_ = np.cos(a), np.sin(a)
    if axis == "x":
        return np.array([[1, 0, 0], [0, c, -s_], [0, s_, c]])
    if axis == "y":
        return np.array([[c, 0, s_], [0, 1, 0], [-s_, 0, c]])
    if axis == "z":
        return np.array([[c, -s_, 0], [s_, c, 0], [0, 0, 1]])
    raise ValueError("axis should be x,y,z")


GENERATIVE_MODELS = ("instantmesh", "trellis", "sf3d")


def reg_points(partial_xyz, complete_xyz, cd_inv_weight=0.5, diff_init=True, reg_fine_xyz=False, dataset="redwood",
               n_fused=20000, lr=0.01, iters=200, partial_rgb=None, complete_rgb=None, generative_model="trellis",
               diff_complete_xyz=None):
    """In-memory form of reg() (reg_xyz.py:99-223): differentiable init -> generator-specific frame fix-up -> 11-scale
    coarse ICP sweep -> optional per-axis scale grid -> fuse (drop generated points that coincide with scan points, FPS to
    n_fused, outlier filter).  partial_xyz = the scan (`color_point.ply`), complete_xyz = the generated shape (163 840
    surface samples in the reference, :125); colours ride along through every selection (:211-219).  diff_complete_xyz:
    the cloud the differentiable init registers (the reference samples the mesh a second time, 120 000 points,
    diff_obj_pose.py:504); default = complete_xyz.  Returns a dict of device tensors.
    Deviations from the reference, all forced by unseeded / unvendored third-party calls (DESIGN.md section 3): FPS
    starts at index 0 (fpsample: random start) and is skipped when the fused cloud already has <= n_fused points."""
    if generative_model not in GENERATIVE_MODELS:
        raise ValueError(f"generative_model {generative_model!r} not supported (reg_xyz.py:133-140 knows {GENERATIVE_MODELS})")
    dev = partial_xyz.device
    source, target = partial_xyz.float(), complete_xyz.float()
    src_rgb = None if partial_rgb is None else partial_rgb.float().to(dev)
    tgt_rgb = None if complete_rgb is None else complete_rgb.float().to(dev)
    diff_T = np.eye(4)
    if diff_init:
        dc = target if diff_complete_xyz is None else diff_complete_xyz.float()
        T = object_pose_optimization_points(voxel_down_sample(dc, 0.02), voxel_down_sample(source, 0.02), lr=lr,
                                            iters=iters, device=dev)
        diff_T = np.linalg.inv(T)                                   # reg_xyz.py:122
    dT = torch.as_tensor(diff_T, dtype=torch.float32, device=dev)
    source = source @ dT[:3, :3].T + dT[:3, 3]                      # partial into the generated shape's frame (:126)
    tn, _, _ = normalize_numpy(target.cpu().numpy(), range=0.5)     # :131
    if generative_model == "instantmesh":                           # :133-138
        keep0 = remove_statistical_outlier(source, 20, 1.5)         # remove_noise_from_point_cloud(source_pcd)
        source = source[keep0]
        src_rgb = None if src_rgb is None else src_rgb[keep0]
        tn = np.dot(np.dot(tn, get_rotate_matrix("x", 90).T), get_rotate_matrix("y", 90).T)
    target = torch.as_tensor(tn, dtype=torch.float32, device=dev)
    # coarse sweep (:146-173), all 11 scales at once
    scales = np.linspace(1.5, 0.8, 11)
    s_down, t_down = voxel_down_sample(source, 0.03), voxel_down_sample(target, 0.03)
    out = coarse_scale_sweep(s_down, t_down, scales, 0.075, cd_inv_weight)
    out["diff_transform"] = diff_T
    coarse = out["coarse_transformation"]
    tgt_full = target
    if reg_fine_xyz:
        source = source @ coarse[:3, :3].T + coarse[:3, 3]          # :176
        s_in = source if dataset in ("pcn", "kitti") else voxel_down_sample(source, 0.03)
        t_in = voxel_down_sample(target, 0.04 if dataset in ("pcn", "kitti") else 0.03)
        Sx, loss_xyz, Txyz = iterative_scale_search(s_in, t_in, [(0.8, 1.2)] * 3, 10, None, cd_inv_weight)
        for Mx in (np.linalg.inv(Sx), np.linalg.inv(Txyz)):         # :194-197
            Mt = torch.as_tensor(Mx, dtype=torch.float32, device=dev)
            tgt_full = tgt_full @ Mt[:3, :3].T + Mt[:3, 3]
        ci = torch.linalg.inv(coarse.double()).float()
        source = source @ ci[:3, :3].T + ci[:3, 3]                  # :199-200
        out.update(best_scales=np.diag(Sx)[:3].copy(), fine_loss=loss_xyz)
    for Mt in (torch.linalg.inv(coarse.double()).float(), torch.as_tensor(np.linalg.inv(diff_T), dtype=torch.float32, device=dev)):
        tgt_full = tgt_full @ Mt[:3, :3].T + Mt[:3, 3]              # :202-205
    di = torch.as_tensor(np.linalg.inv(diff_T), dtype=torch.float32, device=dev)
    source = source @ di[:3, :3].T + di[:3, 3]                      # :206
    keep = remove_close_points(source, tgt_full, 0.0001)            # :210
    fused = torch.cat([source, tgt_full[keep]])                     # :211 fused = source + filtered target
    with_rgb = src_rgb is not None and tgt_rgb is not None
    fused_rgb = torch.cat([src_rgb, tgt_rgb[keep]]) if with_rgb else None
    if fused.shape[0] > n_fused:
        idx = furthest_point_sample(fused[None].contiguous(), n_fused, 0)[0].long()   # :215-217
        fused = fused[idx]
        fused_rgb = fused_rgb[idx] if with_rgb else None
    ok = remove_statistical_outlier(fused, std_ratio=2.5)                             # :219
    fused = fused[ok]
    fused_rgb = fused_rgb[ok] if with_rgb else None
    out.update(fused=fused, fused_rgb=fused_rgb, source=source, target=tgt_full)
    return out
