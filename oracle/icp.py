"""CPU oracle of one point-to-point ICP iteration -- TEST INFRASTRUCTURE ONLY.

Restates what Open3D's registration_icp(TransformationEstimationPointToPoint) does per iteration as the reference calls it
(reg_xyz.py:9-38; Open3D is third-party and not vendored, so this follows its documented algorithm: parity unpinned):
correspondences = nearest neighbour within max_correspondence_distance, fitness = inliers / |source|,
inlier_rmse = sqrt(sum d^2 / inliers), update = the least-squares rigid motion of the inlier pairs by Kabsch / SVD with
the reflection fix (Umeyama without scaling), convergence = both relative changes below the ICPConvergenceCriteria.
csrc/icp.cu reaches the same optimum with Horn's quaternion form; the two agree to double rounding.
"""
import numpy as np


def kabsch(src, dst):
    """Least-squares rigid motion dst ~ R src + t (float64) -> (R [3,3], t [3])."""
    src, dst = np.asarray(src, np.float64), np.asarray(dst, np.float64)
    ms, md = src.mean(0), dst.mean(0)
    H = (src - ms).T @ (dst - md)
    U, _, Vt = np.linalg.svd(H)
    D = np.diag([1.0, 1.0, np.sign(np.linalg.det(Vt.T @ U.T))])
    R = Vt.T @ D @ U.T
    return R, md - R @ ms


def icp_step(cur, target, dist, idx, T, state, max_dist2, rel_fitness, rel_rmse, update=True):
    """One call of genpc_icp_step for ONE candidate.  cur [Ns,3] (source under T), target [Nt,3], dist/idx = squared NN
    distance / index of every cur point, T [4,4] float32, state = [fitness, rmse, converged, calls] float32.
    An inlier has dist < max_dist2 (NaN is none) and an idx in [0, Nt).  -> (T', state')."""
    cur, target = np.asarray(cur, np.float32), np.asarray(target, np.float32)
    dist, idx = np.asarray(dist, np.float32), np.asarray(idx)
    inl = (dist < np.float32(max_dist2)) & (idx >= 0) & (idx < target.shape[0])
    cnt = int(inl.sum())
    fitness = np.float32(cnt / cur.shape[0])
    rmse = np.float32(np.sqrt(dist[inl].astype(np.float64).sum() / (cnt if cnt > 0 else 1)))
    st = np.array(state, np.float32)
    converged = bool(st[2] != 0)
    if not converged and st[3] > 0 and abs(np.float32(fitness - st[0])) < np.float32(rel_fitness) and \
            abs(np.float32(rmse - st[1])) < np.float32(rel_rmse):
        converged = True
    new_state = np.array([fitness, rmse, 1.0 if converged else 0.0, st[3] + 1], np.float32)
    T = np.array(T, np.float32)
    if not update or converged or cnt < 3:
        return T, new_state
    R, t = kabsch(cur[inl], target[idx[inl]])
    M = np.eye(4)
    M[:3, :3], M[:3, 3] = R, t
    Tn = T.copy()
    Tn[:3] = (M @ T.astype(np.float64))[:3].astype(np.float32)
    return Tn, new_state


def icp(source, target, max_dist, max_iteration=30, rel_fitness=1e-6, rel_rmse=1e-6, nn=None):
    """Full loop for one candidate with brute-force float64 nearest neighbours (small clouds only).
    -> (T [4,4] f32, fitness, rmse, iterations run)."""
    source, target = np.asarray(source, np.float32), np.asarray(target, np.float32)
    T = np.eye(4, dtype=np.float32)
    state = np.zeros(4, np.float32)
    for it in range(max_iteration + 1):
        cur = (source @ T[:3, :3].T + T[:3, 3]).astype(np.float32)
        if nn is None:
            d2 = ((cur[:, None, :].astype(np.float64) - target[None].astype(np.float64)) ** 2).sum(-1)
            idx = d2.argmin(1)
            dist = d2[np.arange(len(cur)), idx].astype(np.float32)
        else:
            dist, idx = nn(cur, target)
        T, state = icp_step(cur, target, dist, idx, T, state, max_dist ** 2, rel_fitness, rel_rmse, it < max_iteration)
        if state[2]:
            break
    return T, float(state[0]), float(state[1]), it + 1
