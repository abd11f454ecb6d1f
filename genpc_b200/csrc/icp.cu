// icp.cu -- one point-to-point ICP iteration for K candidates at once (scale / ICP candidate search), sm_100a.
//
// The reference refines every scale candidate with Open3D's registration_icp(TransformationEstimationPointToPoint)
// on the CPU (reg_xyz.py:9-38 inside the 11-candidate sweep :146-173 and the 10x10x10 per-axis grid :60-96; third-party
// code, not vendored).  Here the candidates are the batch dimension: the nearest neighbours of all of them come from ONE
// Chamfer launch (genpc_chamfer_forward), and this kernel does the rest of the iteration for every candidate --
//   inliers (dist < max_dist^2), fitness = inliers / Ns, inlier_rmse = sqrt(sum dist / inliers)   (Open3D's definitions)
//   convergence: |fitness - previous| < rel_fitness and |rmse - previous| < rel_rmse             (ICPConvergenceCriteria)
//   centroids and the 3x3 cross-covariance of the inlier pairs, accumulated in double with a fixed tree (deterministic)
//     about an anchor in the cloud (target row 0), so that clouds far from the origin keep their precision
//   optimal rotation by Horn's closed form: the eigenvector of the largest eigenvalue of the 4x4 matrix N(H) (cyclic
//     Jacobi in double) is the unit quaternion of the rotation that minimises sum |R s + t - q|^2 -- the same optimum
//     Kabsch/SVD with the reflection fix gives, without an SVD;  t = mu_t - R mu_s
//   T <- [R|t] T for candidates that are active and have >= 3 inliers
// -- one CTA per candidate, no host synchronisation anywhere in the loop (the torch formulation it replaces needed ~25
// tiny launches, a batched float64 SVD and one host sync per iteration).  The ragged form (genpc_icp_step_ragged) gives every
// candidate its own source / target point counts and also applies T to the untransformed source, so that a batch of
// differently-sized objects runs one loop.
#include "common.cuh"

namespace genpc {

constexpr int ICP_THREADS = 256;
constexpr int ICP_NACC = 17;  // count, sum s (3), sum q (3), sum s (x) q (9), sum dist

// one Jacobi rotation in the (P, R) plane; every index is a compile-time constant so that A and V stay in registers
// (a first version with run-time p / r loops kept them in local memory: 0.8 ms per call for one thread per candidate)
template <int P, int R>
__device__ __forceinline__ void jacobi_rotate(double (&A)[4][4], double (&V)[4][4]) {
    const double apr = A[P][R];
    if (fabs(apr) < 1e-300) return;
    const double theta = (A[R][R] - A[P][P]) / (2.0 * apr);
    const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
    const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
#pragma unroll
    for (int k = 0; k < 4; ++k) {  // A <- A J
        const double akp = A[k][P], akr = A[k][R];
        A[k][P] = c * akp - s * akr, A[k][R] = s * akp + c * akr;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {  // A <- J^T A
        const double apk = A[P][k], ark = A[R][k];
        A[P][k] = c * apk - s * ark, A[R][k] = s * apk + c * ark;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {  // V <- V J
        const double vkp = V[k][P], vkr = V[k][R];
        V[k][P] = c * vkp - s * vkr, V[k][R] = s * vkp + c * vkr;
    }
}

// largest-eigenvalue eigenvector of a symmetric 4x4 matrix (cyclic Jacobi, double; converges quadratically: 5-7 sweeps)
__device__ __forceinline__ void sym4_top_eigenvector(double (&A)[4][4], double (&q)[4]) {
    double V[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) V[i][j] = (i == j) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 12; ++sweep) {
        const double off = A[0][1] * A[0][1] + A[0][2] * A[0][2] + A[0][3] * A[0][3] + A[1][2] * A[1][2] + A[1][3] * A[1][3] +
                           A[2][3] * A[2][3];
        const double dia = A[0][0] * A[0][0] + A[1][1] * A[1][1] + A[2][2] * A[2][2] + A[3][3] * A[3][3];
        if (off <= 1e-30 * dia || off < 1e-300) break;
        jacobi_rotate<0, 1>(A, V);
        jacobi_rotate<0, 2>(A, V);
        jacobi_rotate<0, 3>(A, V);
        jacobi_rotate<1, 2>(A, V);
        jacobi_rotate<1, 3>(A, V);
        jacobi_rotate<2, 3>(A, V);
    }
    double best = A[0][0];
#pragma unroll
    for (int k = 0; k < 4; ++k) q[k] = V[k][0];
#pragma unroll
    for (int i = 1; i < 4; ++i) {
        const bool take = A[i][i] > best;
        best = take ? A[i][i] : best;
#pragma unroll
        for (int k = 0; k < 4; ++k) q[k] = take ? V[k][i] : q[k];
    }
    const double nrm = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
#pragma unroll
    for (int k = 0; k < 4; ++k) q[k] /= nrm;
}

// cur[j] = T source[j] for j < n, one row per thread in turn: c_r = fma(T[r][2], z, fma(T[r][1], y, fma(T[r][0], x, T[r][3])))
// (DESIGN § 3 item 12), so a candidate's points do not depend on the batch it sits in.  T is read with plain loads: thread 0
// of the CTA may have just written it.
__device__ __forceinline__ void icp_transform_rows(const float *Tk, const float *__restrict__ sp, float *cp, int n) {
    float M[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) M[i] = Tk[i];
    for (int j = threadIdx.x; j < n; j += ICP_THREADS) {
        const float x = __ldg(sp + j * 3), y = __ldg(sp + j * 3 + 1), z = __ldg(sp + j * 3 + 2);
#pragma unroll
        for (int r = 0; r < 3; ++r)
            cp[j * 3 + r] = fmaf(M[r * 4 + 2], z, fmaf(M[r * 4 + 1], y, fmaf(M[r * 4], x, M[r * 4 + 3])));
    }
}

// thread 0: statistics, convergence test and T update of candidate k from the warp partials.  frozen: the candidate entered
// the call converged (ragged form), read nothing and keeps T, fitness and rmse; only its call counter moves.
// The sums are taken about the anchor o (they hold s - o and q - o), so ms / mq below are centroids relative to o.
__device__ __forceinline__ void icp_finish(const double (&sh)[ICP_THREADS / 32][ICP_NACC], const double (&o)[3], float *Tk,
                                           float *st, int *scan_len, int ns, bool frozen, float rel_fitness, float rel_rmse,
                                           int update) {
    if (frozen) {
        st[3] = st[3] + 1.f;
        *scan_len = 0;
        return;
    }
    double a[ICP_NACC];
#pragma unroll
    for (int i = 0; i < ICP_NACC; ++i) {
        double r = 0.0;
#pragma unroll
        for (int w = 0; w < ICP_THREADS / 32; ++w) r += sh[w][i];  // fixed order
        a[i] = r;
    }
    const double cnt = a[0];
    const float fitness = (float)(cnt / (double)(ns > 0 ? ns : 1));
    const float rmse = (float)sqrt(a[16] / (cnt > 0.0 ? cnt : 1.0));
    const bool was_converged = st[2] != 0.f;
    bool converged = was_converged;
    if (!was_converged && st[3] > 0.f && fabsf(fitness - st[0]) < rel_fitness && fabsf(rmse - st[1]) < rel_rmse) converged = true;
    st[0] = fitness, st[1] = rmse, st[2] = converged ? 1.f : 0.f, st[3] = st[3] + 1.f;
    if (scan_len) *scan_len = converged ? 0 : ns;
    if (!update || converged || cnt < 3.0) return;
    // ---- Horn: R from the cross-covariance of the centred inlier pairs ----
    const double ms[3] = {a[1] / cnt, a[2] / cnt, a[3] / cnt}, mq[3] = {a[4] / cnt, a[5] / cnt, a[6] / cnt};
    double H[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) H[r][c] = a[7 + r * 3 + c] - cnt * ms[r] * mq[c];  // sum (s - ms)(q - mq)^T
    double Nm[4][4];
    Nm[0][0] = H[0][0] + H[1][1] + H[2][2];
    Nm[0][1] = H[1][2] - H[2][1], Nm[0][2] = H[2][0] - H[0][2], Nm[0][3] = H[0][1] - H[1][0];
    Nm[1][1] = H[0][0] - H[1][1] - H[2][2];
    Nm[1][2] = H[0][1] + H[1][0], Nm[1][3] = H[2][0] + H[0][2];
    Nm[2][2] = -H[0][0] + H[1][1] - H[2][2];
    Nm[2][3] = H[1][2] + H[2][1];
    Nm[3][3] = -H[0][0] - H[1][1] + H[2][2];
#pragma unroll
    for (int r = 1; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c)
            if (c < r) Nm[r][c] = Nm[c][r];
    double q[4];
    sym4_top_eigenvector(Nm, q);
    const double w = q[0], x = q[1], y = q[2], z = q[3];
    const double R[3][3] = {{1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)},
                            {2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)},
                            {2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)}};
    double t[3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
        t[r] = (mq[r] + o[r]) - (R[r][0] * (ms[0] + o[0]) + R[r][1] * (ms[1] + o[1]) + R[r][2] * (ms[2] + o[2]));
    // ---- T <- [R|t] T ----
    double Told[4][4], Tnew[3][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) Told[r][c] = Tk[r * 4 + c];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c)
            Tnew[r][c] = R[r][0] * Told[0][c] + R[r][1] * Told[1][c] + R[r][2] * Told[2][c] + t[r] * Told[3][c];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) Tk[r * 4 + c] = (float)Tnew[r][c];
}

// One ICP iteration, one CTA per candidate.  Equal-size form (src_len == nullptr, genpc_icp_step): Ns source and Nt target
// points per candidate, source / tgt_len / scan_len unused.  Ragged form (genpc_icp_step_ragged, DESIGN § 3 item 12):
// candidate k has ns = clamp(src_len[k], 0, Ns) source and nt = clamp(tgt_len[Kt == 1 ? 0 : k], 0, Nt) target points; the
// statistics run over j < ns (fitness = inliers / ns), an idx outside [0, nt) is no inlier, a candidate that enters converged
// reads no dist / idx, and once T is final the CTA writes the next iteration's cur = T source for j < ns.  The write is in
// place: only this CTA reads these rows, and all of its reads come before the barrier the write follows.  dist == nullptr:
// transform only (cur and scan_len, state untouched).  A candidate with no points on a side gets no cur row written.
__global__ void __launch_bounds__(ICP_THREADS) icp_step_kernel(float *cur, const float *__restrict__ source,
                                                               const float *__restrict__ target, const float *__restrict__ dist,
                                                               const int *__restrict__ idx, const int *__restrict__ src_len,
                                                               const int *__restrict__ tgt_len, int *scan_len, float *T,
                                                               float *state, int Ns, int Kt, int Nt, float max_dist2,
                                                               float rel_fitness, float rel_rmse, int update) {
    __shared__ double sh[ICP_THREADS / 32][ICP_NACC];
    const int k = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool ragged = src_len != nullptr;
    const int ns = ragged ? min(max(__ldg(src_len + k), 0), Ns) : Ns;
    const int nt = ragged ? min(max(__ldg(tgt_len + (Kt == 1 ? 0 : k)), 0), Nt) : Nt;
    float *st = state + (size_t)k * 4;  // fitness, rmse, converged, calls
    float *Tk = T + (size_t)k * 16;
    if (dist == nullptr) {
        if (tid == 0) scan_len[k] = st[2] != 0.f ? 0 : ns;
        if (nt > 0) icp_transform_rows(Tk, source + (size_t)k * Ns * 3, cur + (size_t)k * Ns * 3, ns);
        return;
    }
    const bool frozen = ragged && st[2] != 0.f;
    const int n = (frozen || nt == 0) ? 0 : ns;
    const float *cp = cur + (size_t)k * Ns * 3;
    const float *tp = target + (size_t)(Kt == 1 ? 0 : k) * Nt * 3;
    const float *dp = dist + (size_t)k * Ns;
    const int *ip = idx + (size_t)k * Ns;
    // anchor o = target row 0 (0 if it is not finite): raw moments about the origin cancel in H = sum s q^T - cnt ms mq^T
    // when the clouds sit far from it (an offset of 1000 at an extent of 0.1 cost 3 fp32 ulps of t), moments about a point
    // of the cloud do not.  It depends on the candidate only, so a candidate's result still does not depend on its batch.
    double o[3] = {0.0, 0.0, 0.0};
    if (n > 0) {
        const float ox = __ldg(tp), oy = __ldg(tp + 1), oz = __ldg(tp + 2);
        if (isfinite(ox) && isfinite(oy) && isfinite(oz)) o[0] = ox, o[1] = oy, o[2] = oz;
    }
    double acc[ICP_NACC];
#pragma unroll
    for (int i = 0; i < ICP_NACC; ++i) acc[i] = 0.0;
    for (int j = tid; j < n; j += ICP_THREADS) {
        const float d = __ldg(dp + j);
        if (!(d < max_dist2)) continue;
        const int t = __ldg(ip + j);
        if ((unsigned)t >= (unsigned)nt) continue;
        const double sx = __ldg(cp + j * 3) - o[0], sy = __ldg(cp + j * 3 + 1) - o[1], sz = __ldg(cp + j * 3 + 2) - o[2];
        const double qx = __ldg(tp + (size_t)t * 3) - o[0], qy = __ldg(tp + (size_t)t * 3 + 1) - o[1],
                     qz = __ldg(tp + (size_t)t * 3 + 2) - o[2];
        acc[0] += 1.0;
        acc[1] += sx, acc[2] += sy, acc[3] += sz;
        acc[4] += qx, acc[5] += qy, acc[6] += qz;
        acc[7] += sx * qx, acc[8] += sx * qy, acc[9] += sx * qz;
        acc[10] += sy * qx, acc[11] += sy * qy, acc[12] += sy * qz;
        acc[13] += sz * qx, acc[14] += sz * qy, acc[15] += sz * qz;
        acc[16] += (double)d;
    }
#pragma unroll
    for (int i = 0; i < ICP_NACC; ++i) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
        if (lane == 0) sh[warp][i] = acc[i];
    }
    __syncthreads();
    if (tid == 0) icp_finish(sh, o, Tk, st, ragged ? scan_len + k : nullptr, ns, frozen, rel_fitness, rel_rmse, update);
    if (!ragged || frozen || ns == 0 || nt == 0) return;
    __syncthreads();  // T is final
    icp_transform_rows(Tk, source + (size_t)k * Ns * 3, cur + (size_t)k * Ns * 3, ns);
}

}  // namespace genpc

using namespace genpc;

extern "C" int genpc_icp_step(const float *cur, const float *target, const float *dist, const int *idx, float *T, float *state,
                              int K, int Ns, int Kt, int Nt, float max_dist2, float rel_fitness, float rel_rmse, int update,
                              genpc_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (K < 0 || Ns <= 0 || Nt <= 0 || (Kt != 1 && Kt != K)) return GENPC_ERR_SHAPE;
    if (K == 0) return GENPC_OK;
    icp_step_kernel<<<(unsigned)K, ICP_THREADS, 0, stream>>>(const_cast<float *>(cur), nullptr, target, dist, idx, nullptr, nullptr,
                                                            nullptr, T, state, Ns, Kt, Nt, max_dist2, rel_fitness, rel_rmse,
                                                            update);
    GENPC_CHECK_LAUNCH();
    return GENPC_OK;
}

extern "C" int genpc_icp_step_ragged(const float *source, float *cur, const float *target, const float *dist, const int *idx,
                                     const int *src_len, const int *tgt_len, int *scan_len, float *T, float *state, int K,
                                     int Ns, int Kt, int Nt, float max_dist2, float rel_fitness, float rel_rmse, int update,
                                     genpc_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!source || !src_len || !tgt_len || !scan_len || (dist == nullptr) != (idx == nullptr)) return GENPC_ERR_SHAPE;
    if (K <= 0 || Ns <= 0 || Nt <= 0 || (Kt != 1 && Kt != K)) return GENPC_ERR_SHAPE;
    icp_step_kernel<<<(unsigned)K, ICP_THREADS, 0, stream>>>(cur, source, target, dist, idx, src_len, tgt_len, scan_len, T, state,
                                                            Ns, Kt, Nt, max_dist2, rel_fitness, rel_rmse, update);
    GENPC_CHECK_LAUNCH();
    return GENPC_OK;
}
