// register.cu -- the Geometric-Preserving-Fusion registration loop: one launch per Adam iteration (small problems)
// or two (large problems, symmetric scan + fix-up/reduce/Adam), never a host synchronisation.
//
// Replaces the Chamfer part of the reference's hot loop (diff_obj_pose.py:518-576):
//     model(return_pts=True)                      :535  -> ObjectPoseOptim.forward :408-436 (transform :419-423)
//     compute_loss_function(...) Chamfer term     :323-334  cd = CDp-L1(pts->ref) + 0.5*CDp-L1(ref->pts); 3.0*cd
//     loss.backward(); optimizer.step(); .item()  :546-548  (2 ext calls = 4 NN scans + 4 grad launches + D2H sync)
// by ONE kernel per iteration that, for every scan (and every multi-start of it):
//   1. applies the current 7-DoF pose on the fly (queries of direction A / targets of direction B): the moving
//      cloud is never materialised;
//   2. runs the two NN scans that are actually needed (the reference runs four) with the shared packed-FP32
//      work item (nn_core.cuh), merging with packed 64-bit atomicMin;
//   3. the last CTA of a scan to finish (atomic ticket) reduces the loss and the 13 pose-gradient scalars
//      (sum g, sum g (x) u, sum g.Ru -- SURVEY.md appendix C; no scatter atomics) in double, deterministically,
//      back-propagates through the Gram-Schmidt 6-D rotation, applies Adam (betas .9/.999, eps 1e-8, three lr
//      groups :524-528), stores the loss, and re-arms the packed buffers for the next launch.
// No host synchronisation anywhere: the 500-iteration loop is 500 back-to-back launches (graph-capturable).
// Large problems (S*Nc*Nr >= 2e8) use the symmetric scan instead (register_sym_scan_kernel: every distance evaluated
// once for both directions, nn_sym.cuh) followed by register_finish_kernel (per-point index fix-up, then the same
// ticketed finalize): two launches per iteration, 1.34x faster at 64 x 16384^2.
// Ragged batches (genpc_register_run_ragged: per-cloud point counts inside padded strides) run register_step_kernel, one
// launch per iteration, whatever the size: each cloud's scans stop at its own counts and its loss is the mean over its own
// points.  The persistent, symmetric and pruned kernels keep their equal-size code (no per-cloud counts there).
#include <cstdlib>
#include <cstring>

#include "nn_core.cuh"
#include "nn_sym.cuh"
#include "nn_prune.cuh"

namespace genpc {

constexpr int REG_NPAR = 10;  // rot_6d[6], trans[3], log_scale[1]

struct RegArgs {
    const float *complete;  // [C][Nc][3] moving clouds (C = S / n_starts)
    const float *center;    // [C][3]     centroid of each moving cloud (register_buffer('center'), :362)
    const float *ref;       // [C][Nr][3] fixed (partial) clouds
    float *params;          // [S][10]
    float *adam_m;          // [S][10]
    float *adam_v;          // [S][10]
    unsigned long long *packedA;  // [S][Nc]
    unsigned long long *packedB;  // [S][Nr]
    int *counters;          // [S]
    double *partials;       // [S][fix_ctas][14] per-CTA loss / gradient partial sums (symmetric path)
    float *loss_hist;       // [S][T]
    int S, n_starts, Nc, Nr, T, t_index;
    int qtilesA, tsplitsA, itemsA, qtilesB, tsplitsB, items_per_scan;
    int rtiles, cspans, span, rows_per_block, fix_ctas, ticket_total;  // symmetric path (rows = ref, cols = moving)
    float step_size[3];     // lr_g / (1 - beta1^t) for the rot / trans / log_scale groups
    float w_fwd, w_inv, cd_weight;
    float omb1, beta2, omb2, eps, bc2_sqrt;  // 1-beta1, beta2, 1-beta2 (rounded from double like torch's scalars)
    // pruned scan (nn_prune.cuh): *select == 0 -> the packed words of both directions already hold exact indices (the symmetric
    // scan kernel returns at once, the finish kernel skips its fix-up); nullptr: exhaustive path only
    const int *select;
    int nn_span;   // targets per work item of the single-launch / persistent kernels (256, 512 or NN_SPAN)
};

// points of `cloud` (clamped to [1, stride] so that no index leaves the cloud whatever a caller passes)
__device__ __forceinline__ int cloud_len(const int *len, int cloud, int stride) {
    return len == nullptr ? stride : min(max(__ldg(len + cloud), 1), stride);
}

__device__ __forceinline__ void load_similarity(const float *par, const float *center, Similarity &T) {
    rot6d_to_matrix(par, T.R);
    T.s = (float)exp((double)par[9]);  // exp in double then rounded: identical on host and device
    T.c[0] = center[0], T.c[1] = center[1], T.c[2] = center[2];
    T.t[0] = par[6], T.t[1] = par[7], T.t[2] = par[8];
}

__device__ __forceinline__ double block_sum(double v, double *sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    double r = 0.0;
    const int nw = blockDim.x >> 5;
    for (int w = 0; w < nw; ++w) r += sh[w];  // fixed order -> deterministic
    return r;
}

// one gradient term: moving point index jm, fixed point index kf, squared distance d, weight coef0 = w/(count)
__device__ __forceinline__ void accum_term(const RegArgs &a, const Similarity &T, const float *V, const float *Rf,
                                           int jm, int kf, float d, double coef0, double *acc) {
    const float sq = __fsqrt_rn(d);
    acc[13] += coef0 * (double)sq;  // loss
    if (!(d > 0.f)) return;         // the reference's sqrt backward is inf/NaN at d == 0 (loss_util.py:37); skipped
    const float *vp = V + (size_t)jm * 3;
    const float ux = __fmul_rn(__fsub_rn(__ldg(vp), T.c[0]), T.s);
    const float uy = __fmul_rn(__fsub_rn(__ldg(vp + 1), T.c[1]), T.s);
    const float uz = __fmul_rn(__fsub_rn(__ldg(vp + 2), T.c[2]), T.s);
    const float rx = __fmaf_rn(T.R[2], uz, __fmaf_rn(T.R[1], uy, __fmul_rn(T.R[0], ux)));
    const float ry = __fmaf_rn(T.R[5], uz, __fmaf_rn(T.R[4], uy, __fmul_rn(T.R[3], ux)));
    const float rz = __fmaf_rn(T.R[8], uz, __fmaf_rn(T.R[7], uy, __fmul_rn(T.R[6], ux)));
    const float px = __fadd_rn(__fadd_rn(rx, T.c[0]), T.t[0]);
    const float py = __fadd_rn(__fadd_rn(ry, T.c[1]), T.t[1]);
    const float pz = __fadd_rn(__fadd_rn(rz, T.c[2]), T.t[2]);
    const float *fp = Rf + (size_t)kf * 3;
    const double coef = coef0 / (double)sq;
    const double gx = coef * (double)__fsub_rn(px, __ldg(fp));
    const double gy = coef * (double)__fsub_rn(py, __ldg(fp + 1));
    const double gz = coef * (double)__fsub_rn(pz, __ldg(fp + 2));
    acc[0] += gx, acc[1] += gy, acc[2] += gz;                                  // dL/dt
    acc[3] += gx * ux, acc[4] += gx * uy, acc[5] += gx * uz;                   // dL/dR (row-major)
    acc[6] += gy * ux, acc[7] += gy * uy, acc[8] += gy * uz;
    acc[9] += gz * ux, acc[10] += gz * uy, acc[11] += gz * uz;
    acc[12] += gx * rx + gy * ry + gz * rz;                                    // dL/dlog_s
}

// Single thread: Gram-Schmidt backward (SURVEY.md appendix C) on the 13 reduced gradient scalars, Adam step, loss record,
// ticket re-armed.  tot = {dL/dt[3], dL/dR[9] row-major, dL/dlog_s, loss}.
// per-iteration Adam scalars (torch.optim.Adam: step_size = lr / (1 - beta1^t), denominator uses sqrt(1 - beta2^t))
struct AdamStep {
    float step_size[3];
    float bc2_sqrt;
    int t_index;
};

__device__ __forceinline__ AdamStep adam_step_from_args(const RegArgs &a) {
    AdamStep st;
    st.step_size[0] = a.step_size[0], st.step_size[1] = a.step_size[1], st.step_size[2] = a.step_size[2];
    st.bc2_sqrt = a.bc2_sqrt, st.t_index = a.t_index;
    return st;
}

__device__ __noinline__ void pose_update(const RegArgs &a, int scan, const Similarity &T, const double *tot, const AdamStep &st) {
    float *par = a.params + (size_t)scan * REG_NPAR;
    float *am = a.adam_m + (size_t)scan * REG_NPAR;
    float *av = a.adam_v + (size_t)scan * REG_NPAR;
    // ---- Gram-Schmidt backward (SURVEY.md appendix C), double ----
    const double a1[3] = {par[0], par[1], par[2]}, a2[3] = {par[3], par[4], par[5]};
    const double b1[3] = {T.R[0], T.R[1], T.R[2]}, b2[3] = {T.R[3], T.R[4], T.R[5]};
    const double G1[3] = {tot[3], tot[4], tot[5]}, G2[3] = {tot[6], tot[7], tot[8]}, G3[3] = {tot[9], tot[10], tot[11]};
    const double n1 = fmax(sqrt(a1[0] * a1[0] + a1[1] * a1[1] + a1[2] * a1[2]), 1e-12);
    const double dp = b1[0] * a2[0] + b1[1] * a2[1] + b1[2] * a2[2];
    const double wv[3] = {a2[0] - dp * b1[0], a2[1] - dp * b1[1], a2[2] - dp * b1[2]};
    const double n2 = fmax(sqrt(wv[0] * wv[0] + wv[1] * wv[1] + wv[2] * wv[2]), 1e-12);
    double H1[3] = {G1[0] + (b2[1] * G3[2] - b2[2] * G3[1]), G1[1] + (b2[2] * G3[0] - b2[0] * G3[2]),
                    G1[2] + (b2[0] * G3[1] - b2[1] * G3[0])};
    const double H2[3] = {G2[0] + (G3[1] * b1[2] - G3[2] * b1[1]), G2[1] + (G3[2] * b1[0] - G3[0] * b1[2]),
                          G2[2] + (G3[0] * b1[1] - G3[1] * b1[0])};
    const double b2H2 = b2[0] * H2[0] + b2[1] * H2[1] + b2[2] * H2[2];
    const double dw[3] = {(H2[0] - b2[0] * b2H2) / n2, (H2[1] - b2[1] * b2H2) / n2, (H2[2] - b2[2] * b2H2) / n2};
    const double b1dw = b1[0] * dw[0] + b1[1] * dw[1] + b1[2] * dw[2];
    const double da2[3] = {dw[0] - b1[0] * b1dw, dw[1] - b1[1] * b1dw, dw[2] - b1[2] * b1dw};
#pragma unroll
    for (int i = 0; i < 3; ++i) H1[i] -= dp * dw[i] + a2[i] * b1dw;
    const double b1H1 = b1[0] * H1[0] + b1[1] * H1[1] + b1[2] * H1[2];
    const double da1[3] = {(H1[0] - b1[0] * b1H1) / n1, (H1[1] - b1[1] * b1H1) / n1, (H1[2] - b1[2] * b1H1) / n1};
    float grad[REG_NPAR] = {(float)da1[0], (float)da1[1], (float)da1[2], (float)da2[0], (float)da2[1], (float)da2[2],
                            (float)tot[0], (float)tot[1], (float)tot[2], (float)tot[12]};
    // ---- Adam (torch.optim.Adam defaults; lr groups of diff_obj_pose.py:524-528), fp32 like torch ----
#pragma unroll
    for (int i = 0; i < REG_NPAR; ++i) {
        const float step = st.step_size[i < 6 ? 0 : (i < 9 ? 1 : 2)];
        const float g = grad[i];
        const float m = am[i] + (g - am[i]) * a.omb1;        // exp_avg.lerp_(grad, 1-beta1)
        const float v = a.beta2 * av[i] + a.omb2 * g * g;    // exp_avg_sq.mul_(beta2).addcmul_(g, g, 1-beta2)
        am[i] = m, av[i] = v;
        const float denom = sqrtf(v) / st.bc2_sqrt + a.eps;
        par[i] = par[i] - step * (m / denom);                // param.addcdiv_(exp_avg, denom, value=-step_size)
    }
    if (a.loss_hist != nullptr) a.loss_hist[(size_t)scan * a.T + st.t_index] = (float)tot[13];
    a.counters[scan] = 0;
}

__device__ __noinline__ void finalize_scan(const RegArgs &a, int scan, const Similarity &T, double *sh, const AdamStep &st) {
    const int cloud = scan / a.n_starts;
    const float *V = a.complete + (size_t)cloud * a.Nc * 3;
    const float *Rf = a.ref + (size_t)cloud * a.Nr * 3;
    unsigned long long *pA = a.packedA + (size_t)scan * a.Nc;
    unsigned long long *pB = a.packedB + (size_t)scan * a.Nr;
    double acc[14];
#pragma unroll
    for (int i = 0; i < 14; ++i) acc[i] = 0.0;
    const double cA = (double)a.cd_weight * (double)a.w_fwd / (double)a.Nc;
    const double cB = (double)a.cd_weight * (double)a.w_inv / (double)a.Nr;
    const int nthr = blockDim.x;
#pragma unroll 4
    for (int j = threadIdx.x; j < a.Nc; j += nthr) {  // direction A: moving point j -> its NN in ref
        const unsigned long long w = __ldcg(pA + j);
        accum_term(a, T, V, Rf, j, (int)(unsigned)(w & 0xffffffffu), __uint_as_float((unsigned)(w >> 32)), cA, acc);
    }
#pragma unroll 4
    for (int k = threadIdx.x; k < a.Nr; k += nthr) {  // direction B: ref point k -> its NN among moving pts
        const unsigned long long w = __ldcg(pB + k);
        accum_term(a, T, V, Rf, (int)(unsigned)(w & 0xffffffffu), k, __uint_as_float((unsigned)(w >> 32)), cB, acc);
    }
    __syncthreads();
    for (int j = threadIdx.x; j < a.Nc; j += nthr) pA[j] = ~0ull;  // re-arm for the next launch
    for (int k = threadIdx.x; k < a.Nr; k += nthr) pB[k] = ~0ull;
    double tot[14];
#pragma unroll
    for (int i = 0; i < 14; ++i) tot[i] = block_sum(acc[i], sh);
    if (threadIdx.x != 0) return;

    pose_update(a, scan, T, tot, st);
}

// A scan of a ragged batch is finalised as an equal-size scan of its own counts: a copy of the arguments whose Nc / Nr are the
// cloud's counts and whose base pointers are moved so that THIS scan's cloud and packed words sit where the stride-based
// addressing of finalize_scan expects them (moved by cloud * (stride - count) points: still inside the buffers).  The loss
// coefficients, loops and re-arm then stop at the counts, and finalize_scan stays the equal-size code.
__device__ __forceinline__ RegArgs cloud_args(const RegArgs &a, const int *nc_len, const int *nr_len, int scan, int cloud) {
    RegArgs b = a;
    const int nc = cloud_len(nc_len, cloud, a.Nc), nr = cloud_len(nr_len, cloud, a.Nr);
    b.complete = a.complete + (size_t)cloud * (a.Nc - nc) * 3;
    b.ref = a.ref + (size_t)cloud * (a.Nr - nr) * 3;
    b.packedA = a.packedA + (size_t)scan * (a.Nc - nc);
    b.packedB = a.packedB + (size_t)scan * (a.Nr - nr);
    b.Nc = nc, b.Nr = nr;
    return b;
}

template <int QT>
// nc_len / nr_len: points of each moving / fixed cloud [C] of a ragged batch (the rest of its Nc / Nr stride is padding that is
// never read); nullptr: every cloud fills its stride.  (Kernel arguments rather than RegArgs fields: the other kernels, which
// take no ragged batches, keep their argument block and code.)
__global__ void __launch_bounds__(NN_THREADS, NN_MINBLOCKS) register_step_kernel(const RegArgs a, const int *nc_len, const int *nr_len) {
    __shared__ __align__(16) float s[3][NN_SPAN];
    __shared__ Similarity T;
    __shared__ int is_last;
    __shared__ double sh[32];
    const int scan = blockIdx.x / a.items_per_scan;
    int item = blockIdx.x - scan * a.items_per_scan;
    const int cloud = scan / a.n_starts;
    if (threadIdx.x == 0) load_similarity(a.params + (size_t)scan * REG_NPAR, a.center + (size_t)cloud * 3, T);
    __syncthreads();
    const float *V = a.complete + (size_t)cloud * a.Nc * 3;
    const float *Rf = a.ref + (size_t)cloud * a.Nr * 3;
    if (nc_len == nullptr) {
        if (item < a.itemsA) {  // A: moving queries vs fixed targets
            const int ts = item % a.tsplitsA, qt = item / a.tsplitsA;
            nn_scan_item<QT>(s, V, a.Nc, qt * (NN_THREADS * QT), Rf, a.Nr, ts * NN_SPAN, 0, &T, nullptr,
                             a.packedA + (size_t)scan * a.Nc);
        } else {                // B: fixed queries vs moving targets
            item -= a.itemsA;
            const int ts = item % a.tsplitsB, qt = item / a.tsplitsB;
            nn_scan_item<QT>(s, Rf, a.Nr, qt * (NN_THREADS * QT), V, a.Nc, ts * NN_SPAN, 0, nullptr, &T,
                             a.packedB + (size_t)scan * a.Nr);
        }
    } else {
        // ragged batch: the grid is sized by the strides, so an item whose query tile or target span lies wholly in the
        // cloud's padding skips the scan -- with no target it would still publish (+inf, out-of-cloud index) -- and only
        // takes its ticket
        const int nc = cloud_len(nc_len, cloud, a.Nc), nr = cloud_len(nr_len, cloud, a.Nr);
        if (item < a.itemsA) {
            const int ts = item % a.tsplitsA, qt = item / a.tsplitsA;
            if (qt * (NN_THREADS * QT) < nc && ts * NN_SPAN < nr)
                nn_scan_item<QT>(s, V, nc, qt * (NN_THREADS * QT), Rf, nr, ts * NN_SPAN, 0, &T, nullptr,
                                 a.packedA + (size_t)scan * a.Nc);
        } else {
            item -= a.itemsA;
            const int ts = item % a.tsplitsB, qt = item / a.tsplitsB;
            if (qt * (NN_THREADS * QT) < nr && ts * NN_SPAN < nc)
                nn_scan_item<QT>(s, Rf, nr, qt * (NN_THREADS * QT), V, nc, ts * NN_SPAN, 0, nullptr, &T,
                                 a.packedB + (size_t)scan * a.Nr);
        }
    }
    // ---- ticket: the last CTA of this scan reduces loss + gradient and steps the optimiser ----
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicAdd(a.counters + scan, 1) == a.items_per_scan - 1);
    __syncthreads();
    if (is_last) {
        __threadfence();
        if (nc_len == nullptr) finalize_scan(a, scan, T, sh, adam_step_from_args(a));
        else finalize_scan(cloud_args(a, nc_len, nr_len, scan, cloud), scan, T, sh, adam_step_from_args(a));
    }
}

// ---- persistent form of the single-launch path: ALL iterations in ONE cooperative launch -----------------------------
// The real pipeline registers 1-3 K-point clouds with 4 starts (diff_obj_pose.py:502-504 after voxel down-sampling): a few
// dozen CTAs per iteration.  With one launch per iteration an iteration costs 37 us (profiles/r01k_registration_small.json),
// and r02 measured that launch latency is NOT what it is made of: a first persistent version that kept the single-CTA
// finalize ran at 36 us -- the chain is scan (7 us) -> ticket -> ONE CTA gathering all Nc + Nr loss / gradient terms with
// dependent L2 round trips (20 us) -> Adam.  Here the grid (one CTA per work item, all co-resident: cooperative launch)
// loops over the iterations on the device and EVERY CTA of a scan takes a slice of the terms:
//   phase 1  scan item -> packed atomicMin                                  | per-scan barrier (monotonic arrival counter)
//   phase 2  this CTA's slice of moving / fixed points: loss + 13 gradient  | ticket: the last CTA adds the per-CTA partials
//            scalars in double, packed words re-armed, partial stored       | in index order (deterministic), steps Adam and
//                                                                           | releases `iter_done[scan] = k + 1`
// Scans never wait for each other.  Adam's per-iteration scalars are computed on the device from t (same double formulas
// as the host loop).
template <int QT, int SPAN = NN_SPAN>
__global__ void __launch_bounds__(NN_THREADS, NN_MINBLOCKS) register_persistent_kernel(RegArgs a, int iters, int t_start, double lr_rot,
                                                                                       double lr_trans, double lr_scale, int *iter_done,
                                                                                       int *arrivals) {
    __shared__ __align__(16) float s[3][SPAN];
    __shared__ Similarity T;
    __shared__ int is_last;
    __shared__ double shp[NN_THREADS / 32][14];
    __shared__ double tot[14];
    const int scan = blockIdx.x / a.items_per_scan;
    const int item0 = blockIdx.x - scan * a.items_per_scan;
    const int n = a.items_per_scan;
    const int cloud = scan / a.n_starts;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float *V = a.complete + (size_t)cloud * a.Nc * 3;
    const float *Rf = a.ref + (size_t)cloud * a.Nr * 3;
    unsigned long long *pA = a.packedA + (size_t)scan * a.Nc;
    unsigned long long *pB = a.packedB + (size_t)scan * a.Nr;
    const int sliceA = (a.Nc + n - 1) / n, sliceB = (a.Nr + n - 1) / n;
    const double cA = (double)a.cd_weight * (double)a.w_fwd / (double)a.Nc;
    const double cB = (double)a.cd_weight * (double)a.w_inv / (double)a.Nr;
    for (int k = 0; k < iters; ++k) {
        if (threadIdx.x == 0) {
            if (k > 0) {   // the pose of iteration k exists once iteration k - 1 of THIS scan has been finalised
                int v;
                for (;;) {
                    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(iter_done + scan) : "memory");
                    if (v >= k) break;
                    __nanosleep(32);
                }
            }
            load_similarity(a.params + (size_t)scan * REG_NPAR, a.center + (size_t)cloud * 3, T);
        }
        __syncthreads();
        // ---- phase 1: this CTA's scan item ----
        int item = item0;
        if (item < a.itemsA) {
            const int ts = item % a.tsplitsA, qt = item / a.tsplitsA;
            nn_scan_item<QT, SPAN>(s, V, a.Nc, qt * (NN_THREADS * QT), Rf, a.Nr, ts * SPAN, 0, &T, nullptr, pA);
        } else {
            item -= a.itemsA;
            const int ts = item % a.tsplitsB, qt = item / a.tsplitsB;
            nn_scan_item<QT, SPAN>(s, Rf, a.Nr, qt * (NN_THREADS * QT), V, a.Nc, ts * SPAN, 0, nullptr, &T, pB);
        }
        // ---- per-scan barrier: every item of the scan has published its minima ----
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) {
            atomicAdd(arrivals + scan, 1);
            const int want = (2 * k + 1) * n;
            int v;
            for (;;) {
                asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(arrivals + scan) : "memory");
                if (v >= want) break;
                __nanosleep(20);
            }
        }
        __syncthreads();
        // ---- phase 2: this CTA's slice of the loss / gradient terms ----
        double acc[14];
#pragma unroll
        for (int i = 0; i < 14; ++i) acc[i] = 0.0;
        for (int j = item0 * sliceA + (int)threadIdx.x; j < min((item0 + 1) * sliceA, a.Nc); j += NN_THREADS) {
            const unsigned long long w = __ldcg(pA + j);
            pA[j] = ~0ull;   // re-armed for the next iteration (nobody touches it before iter_done is released)
            accum_term(a, T, V, Rf, j, (int)(unsigned)(w & 0xffffffffu), __uint_as_float((unsigned)(w >> 32)), cA, acc);
        }
        for (int q = item0 * sliceB + (int)threadIdx.x; q < min((item0 + 1) * sliceB, a.Nr); q += NN_THREADS) {
            const unsigned long long w = __ldcg(pB + q);
            pB[q] = ~0ull;
            accum_term(a, T, V, Rf, (int)(unsigned)(w & 0xffffffffu), q, __uint_as_float((unsigned)(w >> 32)), cB, acc);
        }
#pragma unroll
        for (int i = 0; i < 14; ++i) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
            if (lane == 0) shp[warp][i] = acc[i];
        }
        __syncthreads();
        double *partial = a.partials + ((size_t)scan * n + item0) * 14;
        if (threadIdx.x < 14) {
            double r = 0.0;
#pragma unroll
            for (int w = 0; w < NN_THREADS / 32; ++w) r += shp[w][threadIdx.x];   // fixed order
            partial[threadIdx.x] = r;
            __threadfence();
        }
        __syncthreads();
        if (threadIdx.x == 0) is_last = (atomicAdd(arrivals + scan, 1) == (2 * k + 2) * n - 1);
        __syncthreads();
        if (is_last) {
            __threadfence();
            if (threadIdx.x < 14) {
                double r = 0.0;
                for (int c = 0; c < n; ++c) r += __ldcg(a.partials + ((size_t)scan * n + c) * 14 + threadIdx.x);   // index order
                tot[threadIdx.x] = r;
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                const int t = t_start + k;
                AdamStep st;
                const double bc1 = 1.0 - pow(0.9, (double)(t + 1));
                st.step_size[0] = (float)(lr_rot / bc1), st.step_size[1] = (float)(lr_trans / bc1), st.step_size[2] = (float)(lr_scale / bc1);
                st.bc2_sqrt = (float)sqrt(1.0 - pow(0.999, (double)(t + 1)));
                st.t_index = t;
                pose_update(a, scan, T, tot, st);
                __threadfence();
                asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(iter_done + scan), "r"(k + 1) : "memory");
            }
        }
        __syncthreads();   // T, shp / tot and the staging buffer are free for the next iteration
    }
}

// ---- symmetric path: every distance evaluated once (nn_sym.cuh), two launches per iteration ----------------
// launch 1: rows = fixed cloud (registers), cols = moving cloud (pose applied while staging).
//           packedB[k] <- (dB_k, moving index)  exact;  packedA[j] <- (dA_j, row block of the fixed cloud).
template <int QT>
__global__ void __launch_bounds__(SYM_THREADS, 2) register_sym_scan_kernel(const RegArgs a) {
    __shared__ __align__(16) float s[3][SYM_SPAN_MAX];
    __shared__ Similarity T;
    if (a.select != nullptr && *a.select == 0) return;   // the pruned scan did the work
    const int per_scan = a.rtiles * a.cspans;
    const int scan = blockIdx.x / per_scan;
    const int item = blockIdx.x - scan * per_scan;
    const int cloud = scan / a.n_starts;
    if (threadIdx.x == 0) load_similarity(a.params + (size_t)scan * REG_NPAR, a.center + (size_t)cloud * 3, T);
    __syncthreads();
    const int cs = item % a.cspans, rt = item / a.cspans;
    nn_sym_item<QT>(s, a.ref + (size_t)cloud * a.Nr * 3, a.Nr, rt, a.complete + (size_t)cloud * a.Nc * 3, a.Nc,
                    cs * a.span, a.span, &T, a.packedB + (size_t)scan * a.Nr, a.packedA + (size_t)scan * a.Nc);
}

// launch 2: one warp per moving point resolves its (dist, row block) word to the exact lowest index of the fixed
//           cloud; then EVERY CTA reduces the loss / gradient terms of its own 128 moving points (direction A) and of its
//           slice of the fixed cloud (direction B) to 14 doubles (fixed thread assignment, fixed tree), re-arms the packed
//           words it consumed and stores the partial; the last CTA of a scan (ticket) adds the per-CTA partials in index
//           order -- deterministic -- and steps Adam (pose_update).  (The single-CTA finalize_scan of the small path
//           serialised 32 K gather + double-precision terms per scan: 64 CTAs busy, the rest of the GPU idle.)
constexpr int FIX_THREADS = 512;
// moving points per finish CTA: measured on B200, 64 scans x 16384^2 (profiles/r01i_registration_finish.txt):
// 128 -> 4.41, 256 -> 4.32, 512 -> 4.28 ms per iteration (fewer tickets / partial reductions per point); the largest
// size that still gives every resident-CTA slot (2 per SM) one CTA is used.
static int fix_cols_per_cta(int S, int Nc) {
    for (int cols = 512; cols > 128; cols >>= 1)
        if ((long long)S * ((Nc + cols - 1) / cols) >= 2LL * GENPC_NUM_SMS) return cols;
    return 128;
}
template <int FIX_COLS_PER_CTA>
__global__ void __launch_bounds__(FIX_THREADS, 2) register_finish_kernel(const RegArgs a) {
    __shared__ Similarity T;
    __shared__ int is_last;
    __shared__ double sh[FIX_THREADS / 32][14];
    __shared__ double tot[14];
    const int scan = blockIdx.x / a.fix_ctas;
    const int part = blockIdx.x - scan * a.fix_ctas;
    const int cloud = scan / a.n_starts;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) load_similarity(a.params + (size_t)scan * REG_NPAR, a.center + (size_t)cloud * 3, T);
    __syncthreads();
    const float *V = a.complete + (size_t)cloud * a.Nc * 3;
    const float *Rf = a.ref + (size_t)cloud * a.Nr * 3;
    unsigned long long *pA = a.packedA + (size_t)scan * a.Nc;
    unsigned long long *pB = a.packedB + (size_t)scan * a.Nr;
    const int c_lo = part * FIX_COLS_PER_CTA, c_hi = min(a.Nc, c_lo + FIX_COLS_PER_CTA);
    const bool words_exact = a.select != nullptr && *a.select == 0;
    if (!words_exact) {
        // a warp resolves FIX_COLS_PER_WARP columns (c_lo + warp + k * warps): lane k fetches the word and the transformed
        // point of column k up front (ONE exposed L2 latency for all of them instead of one per column), the columns
        // are then handed round by shuffles and their row-block loads are independent, so they overlap as well
        constexpr int FIX_WARPS = FIX_THREADS / 32, FIX_COLS_PER_WARP = FIX_COLS_PER_CTA / FIX_WARPS;
        static_assert(FIX_COLS_PER_WARP <= 32, "one lane per column");
        const int my_c = c_lo + warp + FIX_WARPS * (lane % FIX_COLS_PER_WARP);
        unsigned long long my_w = 0ull;
        float mx = 0.f, my = 0.f, mz = 0.f;
        if (my_c < c_hi) {
            my_w = __ldcg(pA + my_c);
            mx = __ldg(V + (size_t)my_c * 3), my = __ldg(V + (size_t)my_c * 3 + 1), mz = __ldg(V + (size_t)my_c * 3 + 2);
            apply_similarity(T, mx, my, mz);
        }
#pragma unroll
        for (int k = 0; k < FIX_COLS_PER_WARP; ++k) {
            const int c = c_lo + warp + FIX_WARPS * k;
            if (c >= c_hi) break;  // warp-uniform
            const unsigned long long w = __shfl_sync(0xffffffffu, my_w, k);
            const float x = __shfl_sync(0xffffffffu, mx, k), y = __shfl_sync(0xffffffffu, my, k), z = __shfl_sync(0xffffffffu, mz, k);
            const float d = __uint_as_float((unsigned)(w >> 32));
            if (words_exact) continue;   // warp-uniform
            const int found = sym_fix_column(Rf, a.Nr, a.rows_per_block, x, y, z, d, (int)(unsigned)(w & 0xffffffffu), lane);
            if (lane == 0) pA[c] = pack_dist_idx(d, found);
        }
    }
    __syncthreads();  // the fixed-up words of this CTA's columns are visible to the whole CTA
    // ---- this CTA's share of the loss / gradient terms ----
    double acc[14];
#pragma unroll
    for (int i = 0; i < 14; ++i) acc[i] = 0.0;
    const double cA = (double)a.cd_weight * (double)a.w_fwd / (double)a.Nc;
    const double cB = (double)a.cd_weight * (double)a.w_inv / (double)a.Nr;
    for (int c = c_lo + (int)threadIdx.x; c < c_hi; c += FIX_THREADS) {  // direction A: moving point c -> its NN in ref
        const unsigned long long w = pA[c];
        pA[c] = ~0ull;                                                   // re-arm for the next iteration
        accum_term(a, T, V, Rf, c, (int)(unsigned)(w & 0xffffffffu), __uint_as_float((unsigned)(w >> 32)), cA, acc);
    }
    const int rows_per_cta = (a.Nr + a.fix_ctas - 1) / a.fix_ctas;
    const int k_lo = part * rows_per_cta, k_hi = min(a.Nr, k_lo + rows_per_cta);
    // direction B: fixed point k -> its NN among the moving points; upper threads first so that both directions overlap
    for (int k = k_lo + (FIX_THREADS - 1 - (int)threadIdx.x); k < k_hi; k += FIX_THREADS) {
        const unsigned long long w = __ldcg(pB + k);
        pB[k] = ~0ull;
        accum_term(a, T, V, Rf, (int)(unsigned)(w & 0xffffffffu), k, __uint_as_float((unsigned)(w >> 32)), cB, acc);
    }
#pragma unroll
    for (int i = 0; i < 14; ++i) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
        if (lane == 0) sh[warp][i] = acc[i];
    }
    __syncthreads();
    double *partial = a.partials + ((size_t)scan * a.fix_ctas + part) * 14;
    if (threadIdx.x < 14) {
        double r = 0.0;
#pragma unroll
        for (int w = 0; w < FIX_THREADS / 32; ++w) r += sh[w][threadIdx.x];  // fixed order
        partial[threadIdx.x] = r;
        __threadfence();
    }
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicAdd(a.counters + scan, 1) == a.ticket_total - 1);
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    // ---- last CTA of the scan: partials of all CTAs, in index order ----
    if (warp < 14) {
        const double *pp = a.partials + (size_t)scan * a.fix_ctas * 14 + warp;
        double r = 0.0;
        for (int q0 = 0; q0 < a.fix_ctas; q0 += 32) {  // 32 partials per step: lane tree, then chunks in order
            double v = (q0 + lane < a.fix_ctas) ? __ldcg(pp + (size_t)(q0 + lane) * 14) : 0.0;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            r += v;
        }
        if (lane == 0) tot[warp] = r;
    }
    __syncthreads();
    if (threadIdx.x == 0) pose_update(a, scan, T, tot, adam_step_from_args(a));
}

// current similarity of every scan, for the sort of the moving clouds (pruned path)
__global__ void register_sims_kernel(const RegArgs a, Similarity *sims) {
    const int scan = blockIdx.x * blockDim.x + threadIdx.x;
    if (scan < a.S) load_similarity(a.params + (size_t)scan * REG_NPAR, a.center + (size_t)(scan / a.n_starts) * 3, sims[scan]);
}

}  // namespace genpc

using namespace genpc;

// Pruned scan for the symmetric path (nn_prune.cuh; DESIGN.md section 4.3): the fixed clouds are sorted once per call, the moving
// clouds every iteration in their current pose; default from S * Nc * Nr >= 2^30 evaluations, GENPC_REGISTER_PRUNE=0 / 1 forbids /
// forces it.  Results are those of the exhaustive path bit for bit (same distances, lowest index at the minimum).
static bool register_prune_eligible(int S, int Nc, int Nr) {
    if (Nc < PR_BLOCK || Nr < PR_BLOCK || Nc > PR_MAX_N || Nr > PR_MAX_N) return false;
    const char *k = tunable("GENPC_REGISTER_PRUNE");
    if (k != nullptr) return atoi(k) == 1;
    // measured at 16384 x 16384 (ms per iteration, exhaustive vs pruned): S = 8: 0.57 / 0.89, 16: 1.11 / 1.10, 24: 1.65 / 1.24,
    // 32: 2.19 / 1.48, 64: 4.33 / 2.27 -- the pruned scan has a floor of ~0.7 ms (groups on the unseen side of a shape open every
    // block, one after the other) and needs enough query groups beside them to fill the GPU
    const double groups = (double)S * ((double)Nc + (double)Nr) / PR_GROUP;
    return Nc >= 1024 && Nr >= 1024 && (double)S * (double)Nc * (double)Nr >= (double)(1LL << 30) && groups >= 20000.0;
}

// symmetric path (default for big problems): rows = fixed cloud, cols = moving cloud; the one-scan-per-direction kernel
// stays for tiny fixed clouds and for A/B runs (GENPC_REGISTER_MODE=scan).  Measured on B200
// (profiles/r01d_registration.txt): 64 x 16384^2 -> 5.32 ms/iter (sym) vs 7.12 (scan); tiny problems (2500 x 1000 x 4
// starts) are launch bound and keep the single-launch kernel.
static bool register_takes_sym_path(int S, int Nc, int Nr) {
    const char *mode = tunable("GENPC_REGISTER_MODE");
    const bool big = (double)S * (double)Nc * (double)Nr >= 2e8;
    return (mode == nullptr ? big : strcmp(mode, "sym") == 0) && Nr >= 512;
}

constexpr int REG_SPAN_MIN = 256;   // shortest target span of the persistent kernel's work items

// per-scan slots of 14-double partial sums: one per finish CTA (symmetric path, finest granularity 128 columns) or one per
// work item of the persistent small path (at its finest, one query per thread)
static size_t register_partial_slots(int Nc, int Nr) {
    const size_t fix_ctas = ((size_t)Nc + 128 - 1) / 128;
    const size_t items = (size_t)((Nc + NN_THREADS - 1) / NN_THREADS) * ((Nr + REG_SPAN_MIN - 1) / REG_SPAN_MIN) +
                         (size_t)((Nr + NN_THREADS - 1) / NN_THREADS) * ((Nc + REG_SPAN_MIN - 1) / REG_SPAN_MIN);
    return fix_ctas > items ? fix_ctas : items;
}

// The workspace of S scans of C clouds: packed words, partial sums and counters; for the pruned scan, from the next 256-byte
// boundary, its control words, the scans' similarities and the sorted copies and boxes (side 0: the fixed clouds, side 1: the moving)
struct RegWs {
    size_t bytes;
    RegArgs args;           // packedA, packedB, partials, counters (tickets, iter_done, arrivals)
    int *ctl;
    Similarity *sims;
    PruneSortParams sort;   // sorted records, block and chunk boxes
};
static RegWs register_layout(int S, int C, int Nc, int Nr, bool pruned, void *base = nullptr) {
    WsCursor c{static_cast<char *>(base)};
    RegWs w = {};
    w.args.packedA = c.take<unsigned long long>((size_t)S * Nc);
    w.args.packedB = c.take<unsigned long long>((size_t)S * Nr);
    w.args.partials = c.take<double>((size_t)S * register_partial_slots(Nc, Nr) * 14);
    w.args.counters = c.take<int>(3 * (size_t)S);
    if (!pruned) return w.bytes = c.bytes(), w;
    const int clouds[2] = {C, S}, n[2] = {Nr, Nc};
    c.align_base();
    w.ctl = c.take<int>(4), w.sims = c.take<Similarity>(S, 16);
    w.sort = pr_take_sorted(c, clouds, n);
    return w.bytes = c.bytes(), w;
}

extern "C" size_t genpc_register_workspace_bytes(int S, int Nc, int Nr) {
    if (S < 0 || Nc < 0 || Nr < 0) return 0;
    // (with the pruned scan's extras: sized for one start per cloud -- the largest case; genpc_register_run checks what it needs)
    return register_layout(S, S, Nc, Nr, register_prune_eligible(S, Nc, Nr)).bytes;
}

// Kernel launches one Adam iteration costs at this problem size (1: single-launch path, 2: symmetric scan + finish).
extern "C" int genpc_register_launches_per_iter(int S, int Nc, int Nr) {
    if (S <= 0 || Nc <= 0 || Nr <= 0) return GENPC_ERR_SHAPE;
    if (!register_takes_sym_path(S, Nc, Nr)) return 1;   // (small problems: ONE launch for all iterations of a run call)
    // pruned: similarities, sort of the moving clouds, pruned scan, (de-selected) symmetric scan, finish
    return register_prune_eligible(S, Nc, Nr) ? 5 : 2;
}

// Both entry points.  nc_len / nr_len (device, [C]): points of each cloud for a ragged batch, nullptr for an equal-size one.
// A ragged batch always takes register_step_kernel, one launch per iteration: the persistent, symmetric and pruned kernels
// have no per-cloud sizes (carrying them in the persistent kernel raised its register allocation and cost the equal-size
// small registrations up to 1 us per iteration).
static int register_run(const float *complete, const float *center, const float *ref, const int *nc_len, const int *nr_len,
                        float *params, float *adam_m, float *adam_v, float *loss_hist, int S, int n_starts, int Nc, int Nr,
                        int iters, int t_start, int T, double lr_rot, double lr_trans, double lr_scale, float w_fwd,
                        float w_inv, float cd_weight, void *workspace, size_t workspace_bytes, int reset_workspace,
                        cudaStream_t stream) {
    if (S <= 0 || n_starts <= 0 || S % n_starts != 0 || Nc <= 0 || Nr <= 0 || iters < 0 || t_start < 0) return GENPC_ERR_SHAPE;
    if (loss_hist != nullptr && t_start + iters > T) return GENPC_ERR_SHAPE;
    const int C = S / n_starts;
    if (workspace == nullptr || workspace_bytes < register_layout(S, C, Nc, Nr, false).bytes) return GENPC_ERR_WORKSPACE;
    const bool ragged = nc_len != nullptr;
    const bool sym = !ragged && register_takes_sym_path(S, Nc, Nr);
    const bool prune = sym && register_prune_eligible(S, Nc, Nr) && workspace_bytes >= register_layout(S, C, Nc, Nr, true).bytes;
    const RegWs w = register_layout(S, C, Nc, Nr, prune, workspace);
    RegArgs a = w.args;
    a.complete = complete, a.center = center, a.ref = ref, a.params = params, a.adam_m = adam_m, a.adam_v = adam_v;
    a.loss_hist = loss_hist;
    a.S = S, a.n_starts = n_starts, a.Nc = Nc, a.Nr = Nr, a.T = T;
    // queries per thread of the single-launch path: the real pipeline registers 1-3 K-point clouds with 4 starts -- a few
    // dozen CTAs; fewer queries per thread (more, shorter CTAs) while the grid does not fill the GPU twice over
    int QT = nn_pick_qt(Nc < Nr ? Nc : Nr);
    while (QT > 1) {
        const long long items = (long long)((Nc + NN_THREADS * QT - 1) / (NN_THREADS * QT)) * ((Nr + NN_SPAN - 1) / NN_SPAN) +
                                (long long)((Nr + NN_THREADS * QT - 1) / (NN_THREADS * QT)) * ((Nc + NN_SPAN - 1) / NN_SPAN);
        if ((long long)S * items >= 2LL * GENPC_NUM_SMS) break;
        QT >>= 1;
    }
    // work items of the single-launch kernels for a given target span (NN_SPAN unless the persistent kernel picks a shorter one)
    auto set_span = [&](int span) {
        a.nn_span = span;
        a.qtilesA = (Nc + NN_THREADS * QT - 1) / (NN_THREADS * QT);
        a.tsplitsA = (Nr + span - 1) / span;
        a.itemsA = a.qtilesA * a.tsplitsA;
        a.qtilesB = (Nr + NN_THREADS * QT - 1) / (NN_THREADS * QT);
        a.tsplitsB = (Nc + span - 1) / span;
        a.items_per_scan = a.itemsA + a.qtilesB * a.tsplitsB;
        a.ticket_total = a.items_per_scan;
        return (long long)S * a.items_per_scan;
    };
    long long grid = set_span(NN_SPAN);
    if (grid > 0x7fffffffLL) return GENPC_ERR_RANGE;
    const int SQT = Nr >= 1024 ? 4 : 2;
    long long sgrid = 0, fgrid = 0;
    const int fix_cols = fix_cols_per_cta(S, Nc);
    if (sym) {
        sgrid = sym_tiling(S, Nr, Nc, SQT, a.rtiles, a.span, a.cspans);
        a.rows_per_block = 32 * SQT;
        a.fix_ctas = (Nc + fix_cols - 1) / fix_cols;
        a.ticket_total = a.fix_ctas;
        fgrid = (long long)S * a.fix_ctas;
        if (sgrid > 0x7fffffffLL || fgrid > 0x7fffffffLL) return GENPC_ERR_RANGE;
    }
    a.w_fwd = w_fwd, a.w_inv = w_inv, a.cd_weight = cd_weight;
    a.omb1 = (float)(1.0 - 0.9), a.beta2 = (float)0.999, a.omb2 = (float)(1.0 - 0.999), a.eps = (float)1e-8;
    if (reset_workspace) {
        cudaError_t e = cudaMemsetAsync(a.packedA, 0xff, ((size_t)S * Nc + (size_t)S * Nr) * 8, stream);
        if (e != cudaSuccess) return (int)e;
        e = cudaMemsetAsync(a.counters, 0, (size_t)S * sizeof(int), stream);
        if (e != cudaSuccess) return (int)e;
    }
    // ---- small problems: one cooperative launch runs all the iterations (register_persistent_kernel) ----
    if (!sym && !ragged && iters > 1) {
        const char *pk = tunable("GENPC_REGISTER_PERSIST");
        int dev = 0, sms = 0, per_sm = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaError_t eo = cudaSuccess;
        switch (QT) {
            case 4: eo = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, register_persistent_kernel<4>, NN_THREADS, 0); break;
            case 2: eo = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, register_persistent_kernel<2>, NN_THREADS, 0); break;
            default: eo = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, register_persistent_kernel<1>, NN_THREADS, 0); break;
        }
        // shorter target spans spread a scan over more CTAs (the scan phase is the longest link of an iteration's chain): the
        // shortest of 256 / 512 / NN_SPAN whose grid is still co-resident, when the fixed cloud fits one full span (the real
        // pipeline's 1 K-point scans).  Same-box A/B (us per iteration, 4 starts): 1200 x 800 25.2 -> 19.8, 2500 x 1000 25.8 ->
        // 23.7; with a larger fixed cloud the extra merges cost more than the shorter scans save (924 x 2500: 25.4 -> 27.1), so
        // those keep full spans.  The results do not depend on the split (packed atomicMin merge).
        if (eo == cudaSuccess && (pk == nullptr || atoi(pk) != 0) && QT == 1 && Nr <= NN_SPAN) {
            for (int span = REG_SPAN_MIN; span < NN_SPAN; span <<= 1) {
                if (set_span(span) <= (long long)sms * per_sm) break;
                set_span(NN_SPAN);
            }
            grid = (long long)S * a.items_per_scan;
        }
        if (eo == cudaSuccess && (pk == nullptr || atoi(pk) != 0) && grid <= (long long)sms * per_sm) {
            int *iter_done = a.counters + S, *arrivals = a.counters + 2 * S;
            cudaError_t e = cudaMemsetAsync(iter_done, 0, 2 * (size_t)S * sizeof(int), stream);
            if (e != cudaSuccess) return (int)e;
            int it_n = iters, t0 = t_start;
            void *kargs[] = {(void *)&a, (void *)&it_n, (void *)&t0, (void *)&lr_rot, (void *)&lr_trans, (void *)&lr_scale, (void *)&iter_done,
                             (void *)&arrivals};
            const void *fn = QT == 4 ? (const void *)register_persistent_kernel<4>
                                     : (QT == 2 ? (const void *)register_persistent_kernel<2>
                                                : (a.nn_span == 256 ? (const void *)register_persistent_kernel<1, 256>
                                                                    : (a.nn_span == 512 ? (const void *)register_persistent_kernel<1, 512>
                                                                                        : (const void *)register_persistent_kernel<1>)));
            e = cudaLaunchCooperativeKernel(fn, dim3((unsigned)grid), dim3(NN_THREADS), kargs, 0, stream);
            if (e != cudaSuccess) return (int)e;
            return GENPC_OK;
        }
        grid = set_span(NN_SPAN);   // not co-resident: one launch per iteration with full spans
    }
    // ---- pruned scan set-up: control words, similarities, sorted copies behind the base workspace ----
    PruneSortParams sp = w.sort;
    PrunePair pp = {};
    if (prune) {
        cudaError_t e = cudaMemsetAsync(w.ctl, 0, 16, stream);
        if (e != cudaSuccess) return (int)e;
        sp.xyz[0] = ref, sp.xyz[1] = complete, sp.limit = 1e15f, sp.ctl = w.ctl, sp.hilbert = 1;
        sp.single_side = 1, sp.accumulate = 1;
        // the fixed clouds once per call (their verdict opens the flag), the moving clouds every iteration (OR-ed in)
        sp.side0 = 0, sp.B = C, sp.accumulate = 0;
        nn_bin_sort_kernel<1><<<C, PR_SORT_THREADS, 0, stream>>>(sp);
        GENPC_CHECK_LAUNCH();
        sp.side0 = 1, sp.B = S, sp.accumulate = 1, sp.src_div[1] = n_starts, sp.sim[1] = w.sims;
        a.select = w.ctl + 1;
        PruneParams qa = {}, qb = {};
        qa.B = S, qa.select = w.ctl + 1;
        qb = qa;
        // direction A: moving point -> nearest fixed point (packedA); direction B: fixed point -> nearest moving point (packedB)
        qa.q = sp.sorted[1], qa.t = sp.sorted[0], qa.tbox = sp.boxes[0], qa.tcbox = sp.cboxes[0], qa.out = a.packedA, qa.nq = Nc, qa.nt = Nr;
        qa.qdiv = 1, qa.tdiv = n_starts;
        qb.q = sp.sorted[0], qb.t = sp.sorted[1], qb.tbox = sp.boxes[1], qb.tcbox = sp.cboxes[1], qb.out = a.packedB, qb.nq = Nr, qb.nt = Nc;
        qb.qdiv = n_starts, qb.tdiv = 1;
        pp = pr_pair(qa, qb);
    }
    for (int it = 0; it < iters; ++it) {
        const int t = t_start + it;
        a.t_index = t;
        const double bc1 = 1.0 - pow(0.9, (double)(t + 1));
        a.step_size[0] = (float)(lr_rot / bc1), a.step_size[1] = (float)(lr_trans / bc1), a.step_size[2] = (float)(lr_scale / bc1);
        a.bc2_sqrt = (float)sqrt(1.0 - pow(0.999, (double)(t + 1)));
        if (sym) {
            if (prune) {
                register_sims_kernel<<<(S + 127) / 128, 128, 0, stream>>>(a, w.sims);
                nn_bin_sort_kernel<1><<<S, PR_SORT_THREADS, 0, stream>>>(sp);
                pr_launch(pp, stream);
                GENPC_CHECK_LAUNCH();
            }
            if (SQT == 4) register_sym_scan_kernel<4><<<(unsigned)sgrid, SYM_THREADS, 0, stream>>>(a);
            else register_sym_scan_kernel<2><<<(unsigned)sgrid, SYM_THREADS, 0, stream>>>(a);
            GENPC_CHECK_LAUNCH();
            if (fix_cols == 512) register_finish_kernel<512><<<(unsigned)fgrid, FIX_THREADS, 0, stream>>>(a);
            else if (fix_cols == 256) register_finish_kernel<256><<<(unsigned)fgrid, FIX_THREADS, 0, stream>>>(a);
            else register_finish_kernel<128><<<(unsigned)fgrid, FIX_THREADS, 0, stream>>>(a);
            GENPC_CHECK_LAUNCH();
            continue;
        }
        switch (QT) {
            case 4: register_step_kernel<4><<<(unsigned)grid, NN_THREADS, 0, stream>>>(a, nc_len, nr_len); break;
            case 2: register_step_kernel<2><<<(unsigned)grid, NN_THREADS, 0, stream>>>(a, nc_len, nr_len); break;
            default: register_step_kernel<1><<<(unsigned)grid, NN_THREADS, 0, stream>>>(a, nc_len, nr_len); break;
        }
        GENPC_CHECK_LAUNCH();
    }
    return GENPC_OK;
}

extern "C" int genpc_register_run(const float *complete, const float *center, const float *ref, float *params,
                                  float *adam_m, float *adam_v, float *loss_hist, int S, int n_starts, int Nc, int Nr,
                                  int iters, int t_start, int T, double lr_rot, double lr_trans, double lr_scale,
                                  float w_fwd, float w_inv, float cd_weight, void *workspace, size_t workspace_bytes,
                                  int reset_workspace, genpc_stream_t stream) {
    return register_run(complete, center, ref, nullptr, nullptr, params, adam_m, adam_v, loss_hist, S, n_starts, Nc, Nr, iters,
                        t_start, T, lr_rot, lr_trans, lr_scale, w_fwd, w_inv, cd_weight, workspace, workspace_bytes,
                        reset_workspace, (cudaStream_t)stream);
}

extern "C" int genpc_register_run_ragged(const float *complete, const float *center, const float *ref, const int *complete_len,
                                         const int *ref_len, float *params, float *adam_m, float *adam_v, float *loss_hist,
                                         int S, int n_starts, int Nc, int Nr, int iters, int t_start, int T, double lr_rot,
                                         double lr_trans, double lr_scale, float w_fwd, float w_inv, float cd_weight,
                                         void *workspace, size_t workspace_bytes, int reset_workspace, genpc_stream_t stream) {
    if (complete_len == nullptr || ref_len == nullptr) return GENPC_ERR_SHAPE;
    return register_run(complete, center, ref, complete_len, ref_len, params, adam_m, adam_v, loss_hist, S, n_starts, Nc, Nr,
                        iters, t_start, T, lr_rot, lr_trans, lr_scale, w_fwd, w_inv, cd_weight, workspace, workspace_bytes,
                        reset_workspace, (cudaStream_t)stream);
}
