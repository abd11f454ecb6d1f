"""CPU oracle for the GenPC geometric hot path -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this package, and only as the checker / CPU baseline.  genpc_b200/ never does.

numpy-in / numpy-out wrappers over oracle/libgenpc_oracle.so (oracle/genpc_oracle.c, which cites the
reference file:line each function follows), plus loaders for the unmodified reference CUDA extensions
built into oracle/_ref/ (GPU box only).
"""
import ctypes
import importlib.util
import os

import numpy as np

from . import build as _build

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None

_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
_u64p = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")
_int = ctypes.c_int
_flt = ctypes.c_float
_vp = ctypes.c_void_p


def lib():
    global _lib
    if _lib is None:
        so = _build.build_oracle()
        L = ctypes.CDLL(so)
        L.oracle_nn_distance.argtypes = [_int, _int, _f32p, _int, _f32p, _f32p, _i32p]
        L.oracle_chamfer_forward.argtypes = [_int, _int, _int, _f32p, _f32p, _f32p, _f32p, _i32p, _i32p]
        L.oracle_chamfer_backward.argtypes = [_int, _int, _int, _f32p, _f32p, _f32p, _f32p, _i32p, _i32p,
                                              _f32p, _f32p]
        L.oracle_emd_forward.argtypes = [_int, _int, _int, _f32p, _f32p, _f32p, _i32p, _f32p, _i32p, _i32p,
                                         _f32p, _f32p, _i32p, _i32p, _flt, _int]
        L.oracle_emd_forward.restype = _int
        L.oracle_emd_backward.argtypes = [_int, _int, _f32p, _f32p, _f32p, _i32p, _f32p]
        L.oracle_fps.argtypes = [_int, _int, _int, _int, _f32p, _i32p, _vp]
        L.oracle_knn_mean_distance.argtypes = [_int, _int, _int, _f32p, _f32p]
        L.oracle_project_uv.argtypes = [_int, _int, _f32p, _f32p, _int, _flt, _f32p, _f32p, _f32p]
        L.oracle_zbuffer.argtypes = [_int, _int, _int, _int, _f32p, _f32p, _vp, _u64p]
        L.oracle_zbuffer_resolve.argtypes = [_int, _int, _int, _u64p, _f32p, _f32p, _i32p, _f32p]
        L.oracle_unproject.argtypes = [_int, _int, _int, _f32p, _f32p, _int, _u64p, _f32p, _f32p, _i32p,
                                       _i32p]
        L.oracle_pose_matrix.argtypes = [_f32p, _f32p]
        L.oracle_transform.argtypes = [_int, _f32p, _f32p, _f32p, _f32p]
        L.oracle_fmaf.argtypes = [_int, _f32p, _f32p, _f32p, _f32p]
        _lib = L
    return _lib


def _c(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


def chamfer_forward(xyz1, xyz2):
    """(dist1[B,N], dist2[B,M], idx1[B,N] i32, idx2[B,M] i32) -- chamfer3D.cu:12-154."""
    xyz1, xyz2 = _c(xyz1, np.float32), _c(xyz2, np.float32)
    B, N, _ = xyz1.shape
    M = xyz2.shape[1]
    d1 = np.zeros((B, N), np.float32)
    d2 = np.zeros((B, M), np.float32)
    i1 = np.zeros((B, N), np.int32)
    i2 = np.zeros((B, M), np.int32)
    lib().oracle_chamfer_forward(B, N, M, xyz1, xyz2, d1, d2, i1, i2)
    return d1, d2, i1, i2


def nn_distance(q, t):
    """One direction only: (dist[B,N], idx[B,N])."""
    q, t = _c(q, np.float32), _c(t, np.float32)
    B, N, _ = q.shape
    M = t.shape[1]
    d = np.zeros((B, N), np.float32)
    i = np.zeros((B, N), np.int32)
    lib().oracle_nn_distance(B, N, q, M, t, d, i)
    return d, i


def chamfer_backward(xyz1, xyz2, g1, g2, i1, i2):
    """(gradxyz1, gradxyz2) -- chamfer3D.cu:155-195, double-accumulated."""
    xyz1, xyz2 = _c(xyz1, np.float32), _c(xyz2, np.float32)
    B, N, _ = xyz1.shape
    M = xyz2.shape[1]
    gx1 = np.zeros((B, N, 3), np.float32)
    gx2 = np.zeros((B, M, 3), np.float32)
    lib().oracle_chamfer_backward(B, N, M, xyz1, xyz2, _c(g1, np.float32), _c(g2, np.float32),
                                  _c(i1, np.int32), _c(i2, np.int32), gx1, gx2)
    return gx1, gx2


def emd_forward(xyz1, xyz2, eps, iters, return_state=False, getmax_lowest=False):
    """(dist[B,n], assignment[B,n]) -- emd_cuda.cu:228-282 with emd_module.py:43-54 initial state.
    getmax_lowest: resolve the reference's GetMax store race (:188-191) as "lowest bidder index wins" instead of the
    default "highest" (both are legitimate outcomes of the race; see the comment in genpc_oracle.c)."""
    xyz1, xyz2 = _c(xyz1, np.float32), _c(xyz2, np.float32)
    B, n, _ = xyz1.shape
    m = xyz2.shape[1]
    dist = np.zeros((B, n), np.float32)
    asg = np.full((B, n), -1, np.int32)
    asg_inv = np.full((B, m), -1, np.int32)
    price = np.zeros((B, m), np.float32)
    bid = np.zeros((B, n), np.int32)
    binc = np.zeros((B, n), np.float32)
    minc = np.zeros((B, m), np.float32)
    uidx = np.zeros(B * n, np.int32)
    midx = np.zeros(B * m, np.int32)
    lib().oracle_emd_set_getmax_rule(1 if getmax_lowest else 0)
    try:
        rc = lib().oracle_emd_forward(B, n, m, xyz1, xyz2, dist, asg, price, asg_inv, bid, binc, minc, uidx,
                                      midx, float(eps), int(iters))
    finally:
        lib().oracle_emd_set_getmax_rule(0)
    if rc != 1:
        raise ValueError(f"oracle_emd_forward rejected the shapes (rc={rc})")
    if return_state:
        return dist, asg, dict(price=price, assignment_inv=asg_inv, bid=bid, bid_increments=binc,
                               max_increments=minc, max_idx=midx)
    return dist, asg


def emd_backward(xyz1, xyz2, graddist, assignment):
    xyz1, xyz2 = _c(xyz1, np.float32), _c(xyz2, np.float32)
    B, n, _ = xyz1.shape
    g = np.zeros((B, n, 3), np.float32)
    lib().oracle_emd_backward(B, n, xyz1, xyz2, _c(graddist, np.float32), _c(assignment, np.int32), g)
    return g


def fps(xyz, K, start=0, return_seq=False):
    """idx[B,K] i32 (and the selected-distance sequence) -- semantics defined in genpc_oracle.c."""
    xyz = _c(xyz, np.float32)
    B, N, _ = xyz.shape
    idx = np.zeros((B, K), np.int32)
    seq = np.zeros((B, K), np.float32)
    lib().oracle_fps(B, N, K, int(start), xyz, idx, seq.ctypes.data_as(_vp))
    return (idx, seq) if return_seq else idx


def knn_mean_distance(xyz, k, include_self=True):
    """mean distance to the k nearest neighbours of each point of xyz [N,3] (Open3D remove_statistical_outlier's
    per-point statistic, reg_xyz.py:219); float32 [N]."""
    xyz = _c(xyz, np.float32)
    if not 1 <= k <= 32:
        raise ValueError("1 <= k <= 32")
    out = np.zeros(xyz.shape[0], np.float32)
    lib().oracle_knn_mean_distance(xyz.shape[0], int(k), int(bool(include_self)), xyz, out)
    return out


def statistical_outlier_mask(mean_dist, std_ratio):
    """Open3D's threshold over the per-point means (float64 like its std::vector<double>): keep a point when
    0 < mean < cloud_mean + std_ratio * std_dev.  As in Open3D's RemoveStatisticalOutliers, only means > 0 enter the two
    sums, while the divisors count every point whose query found something (mean >= 0): cloud_mean = sum / n_valid,
    std_dev = sqrt(sum((mean - cloud_mean)^2 over mean > 0) / (n_valid - 1))."""
    m = np.asarray(mean_dist, np.float64)
    nv = int((m >= 0).sum())
    if nv == 0:
        return np.zeros(m.shape, bool)
    pos = m > 0
    mu = m[pos].sum() / nv
    sd = np.sqrt(((m[pos] - mu) ** 2).sum() / (nv - 1)) if nv > 1 else 0.0
    return pos & (m < mu + std_ratio * sd)


def project_uv(cams, xyz, rescale=True, padding=0.15):
    """cams[V,16], xyz[N,3] -> ndc[V,N,3], uv[V,N,2], bounds[V,4] -- DepthPrompting.py:239-271."""
    cams, xyz = _c(cams, np.float32), _c(xyz, np.float32)
    V, N = cams.shape[0], xyz.shape[0]
    ndc = np.zeros((V, N, 3), np.float32)
    uv = np.zeros((V, N, 2), np.float32)
    bounds = np.zeros((V, 4), np.float32)
    lib().oracle_project_uv(V, N, cams, xyz, int(bool(rescale)), float(padding), ndc, uv, bounds)
    return ndc, uv, bounds


def zbuffer(uv, ndc, res, point_size=1, valid=None):
    """packed z-buffer[V,res,res] u64 -- DepthPrompting.py:179-184, 292-339 + defined depth test."""
    uv, ndc = _c(uv, np.float32), _c(ndc, np.float32)
    V, N = uv.shape[0], uv.shape[1]
    zb = np.zeros((V, res, res), np.uint64)
    vp = None
    if valid is not None:
        valid = _c(valid, np.uint8)
        vp = valid.ctypes.data_as(_vp)
    lib().oracle_zbuffer(V, N, res, int(point_size), uv, ndc, vp, zb)
    return zb


def zbuffer_resolve(zb, ndc, zminmax):
    zb, ndc = _c(zb, np.uint64), _c(ndc, np.float32)
    V, res = zb.shape[0], zb.shape[1]
    N = ndc.shape[1]
    idx = np.zeros((V, res, res), np.int32)
    dep = np.zeros((V, res, res), np.float32)
    lib().oracle_zbuffer_resolve(V, N, res, zb, ndc, _c(zminmax, np.float32), idx, dep)
    return idx, dep


def unproject(cams, bounds, zb, ndc, rescale=True):
    cams, bounds, zb, ndc = _c(cams, np.float32), _c(bounds, np.float32), _c(zb, np.uint64), _c(ndc, np.float32)
    V, res = zb.shape[0], zb.shape[1]
    N = ndc.shape[1]
    out = np.zeros((V, res * res, 3), np.float32)
    own = np.zeros((V, res * res), np.int32)
    counts = np.zeros(V, np.int32)
    lib().oracle_unproject(V, N, res, cams, bounds, int(bool(rescale)), zb, ndc, out, own, counts)
    return out, own, counts


def pose_matrix(rot6d):
    """rotation_6d_to_matrix with explicit fp32 rounding -> R [3,3] float32."""
    R = np.zeros(9, np.float32)
    lib().oracle_pose_matrix(_c(rot6d, np.float32), R)
    return R.reshape(3, 3)


def transform(V, center, params):
    """pts = R (s (V - c)) + c + t, params = rot6d[6] | trans[3] | log_scale[1] (diff_obj_pose.py:419-423)."""
    V = _c(V, np.float32)
    out = np.zeros_like(V)
    lib().oracle_transform(V.shape[0], V, _c(center, np.float32), _c(params, np.float32), out)
    return out


def fmaf(a, b, c):
    """fp32 a * b + c with one rounding (C fmaf), elementwise with numpy broadcasting -> float32 array."""
    a, b, c = (_c(x, np.float32) for x in np.broadcast_arrays(*(np.asarray(x, np.float32) for x in (a, b, c))))
    out = np.zeros(a.shape, np.float32)
    lib().oracle_fmaf(a.size, a, b, c, out)
    return out


# ----------------------------------------------------------------------------------------------------
# The unmodified reference extensions (GPU only; built by oracle/build.py into oracle/_ref/).
# ----------------------------------------------------------------------------------------------------
def load_ref_ext(name):
    """Import oracle/_ref/<name>/<name>.so (pybind module `chamfer_3D` or `emd`); None if not built."""
    so = _build.ref_so_path(name)
    if not os.path.exists(so):
        return None
    import torch  # noqa: F401  (the extension links against libtorch)

    spec = importlib.util.spec_from_file_location(name, so)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod
