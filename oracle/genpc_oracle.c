/*
 * genpc_oracle.c -- CPU restatement of GenPC's geometric hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is imported, linked or executed by the
 * product (genpc_b200/).  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs may use it, and only as the checker / the CPU baseline.
 *
 * Parity status:
 *   - Chamfer forward/backward, EMD: restated from the reference's CUDA sources (cited per function).
 *     The reference ships no golden vectors and no CPU implementation; the restatement is pinned on the
 *     GPU box against the UNMODIFIED reference extensions built into oracle/_ref/ (tests/test_ref_ext_gpu.py).
 *   - FPS, projection, z-buffer, unprojection: the arithmetic lives in un-vendored third-party packages
 *     (fpsample, kaolin, open3d) or does not exist in the reference at all -> "parity unpinned";
 *     this file DEFINES the semantics (DESIGN.md section 3).
 *
 * Build: see oracle/build.py  (gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC).
 * Every floating-point contraction is written explicitly with fmaf(); -ffp-contract=off forbids others.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#if defined(__x86_64__)
#define HOT __attribute__((target_clones("fma", "default")))
#else
#define HOT
#endif

/* Squared distance exactly as nvcc contracts `x2*x2+y2*y2+z2*z2` (chamfer3D.cu:35, -fmad=true):
 * fma(dz,dz, fma(dx,dx, dy*dy)) with d* = target - query  (SURVEY.md section 2b, PTX probe). */
static inline float sqdist_ref(float qx, float qy, float qz, float tx, float ty, float tz) {
    float dx = tx - qx, dy = ty - qy, dz = tz - qz;
    return fmaf(dz, dz, fmaf(dx, dx, dy * dy));
}

/* ------------------------------------------------------------------------------------------------
 * Chamfer forward, one direction.  Follows NmDistanceKernel (chamfer3D.cu:12-134):
 * targets are visited in chunks of 512; inside a chunk slot 0 is taken unconditionally and later
 * slots win on strict `d<best` (:36,:46); across chunks the running result is replaced on strict
 * `result>best` (:126).  For finite inputs this is "global min, lowest index on ties".
 * ---------------------------------------------------------------------------------------------- */
HOT void oracle_nn_distance(int b, int n, const float *xyz, int m, const float *xyz2, float *result,
                            int *result_i) {
    const int batch = 512;
#pragma omp parallel for schedule(static) collapse(2)
    for (int i = 0; i < b; i++) {
        for (int j = 0; j < n; j++) {
            const float x1 = xyz[((size_t)i * n + j) * 3 + 0];
            const float y1 = xyz[((size_t)i * n + j) * 3 + 1];
            const float z1 = xyz[((size_t)i * n + j) * 3 + 2];
            float res = 0.f;
            int res_i = 0;
            for (int k2 = 0; k2 < m; k2 += batch) {
                int end_k = (m < k2 + batch ? m : k2 + batch) - k2;
                const float *buf = xyz2 + ((size_t)i * m + k2) * 3;
                float best = 0.f;
                int best_i = 0;
                for (int k = 0; k < end_k; k++) {
                    float d = sqdist_ref(x1, y1, z1, buf[k * 3 + 0], buf[k * 3 + 1], buf[k * 3 + 2]);
                    if (k == 0 || d < best) {
                        best = d;
                        best_i = k + k2;
                    }
                }
                if (k2 == 0 || res > best) {
                    res = best;
                    res_i = best_i;
                }
            }
            result[(size_t)i * n + j] = res;
            result_i[(size_t)i * n + j] = res_i;
        }
    }
}

/* chamfer_cuda_forward (chamfer3D.cu:136-154): both directions. */
void oracle_chamfer_forward(int B, int N, int M, const float *xyz1, const float *xyz2, float *dist1,
                            float *dist2, int *idx1, int *idx2) {
    oracle_nn_distance(B, N, xyz1, M, xyz2, dist1, idx1);
    oracle_nn_distance(B, M, xyz2, N, xyz1, dist2, idx2);
}

/* ------------------------------------------------------------------------------------------------
 * Chamfer backward.  Follows NmDistanceGradKernel (chamfer3D.cu:155-174) launched twice (:184-185).
 * Each term is formed in fp32 exactly as the reference does (g = grad*2; g*(x1-x2), no contraction
 * possible); the reference then accumulates with unordered float atomics, so its sum is not
 * reproducible -- the oracle accumulates the fp32 terms in double and rounds once ("truth" for the
 * 1e-5 relative check).  acc1/acc2 are caller-provided double scratch [B*N*3], [B*M*3], zeroed here.
 * ---------------------------------------------------------------------------------------------- */
static void grad_one_direction(int b, int n, const float *xyz1, int m, const float *xyz2,
                               const float *grad_dist1, const int *idx1, double *acc1, double *acc2) {
    for (int i = 0; i < b; i++) {
        for (int j = 0; j < n; j++) {
            float x1 = xyz1[((size_t)i * n + j) * 3 + 0];
            float y1 = xyz1[((size_t)i * n + j) * 3 + 1];
            float z1 = xyz1[((size_t)i * n + j) * 3 + 2];
            int j2 = idx1[(size_t)i * n + j];
            float x2 = xyz2[((size_t)i * m + j2) * 3 + 0];
            float y2 = xyz2[((size_t)i * m + j2) * 3 + 1];
            float z2 = xyz2[((size_t)i * m + j2) * 3 + 2];
            float g = grad_dist1[(size_t)i * n + j] * 2;
            float tx = g * (x1 - x2), ty = g * (y1 - y2), tz = g * (z1 - z2);
            acc1[((size_t)i * n + j) * 3 + 0] += tx;
            acc1[((size_t)i * n + j) * 3 + 1] += ty;
            acc1[((size_t)i * n + j) * 3 + 2] += tz;
            acc2[((size_t)i * m + j2) * 3 + 0] += -tx;
            acc2[((size_t)i * m + j2) * 3 + 1] += -ty;
            acc2[((size_t)i * m + j2) * 3 + 2] += -tz;
        }
    }
}

void oracle_chamfer_backward(int B, int N, int M, const float *xyz1, const float *xyz2,
                             const float *graddist1, const float *graddist2, const int *idx1,
                             const int *idx2, float *gradxyz1, float *gradxyz2) {
    size_t n1 = (size_t)B * N * 3, n2 = (size_t)B * M * 3;
    double *acc1 = (double *)calloc(n1 ? n1 : 1, sizeof(double));
    double *acc2 = (double *)calloc(n2 ? n2 : 1, sizeof(double));
    grad_one_direction(B, N, xyz1, M, xyz2, graddist1, idx1, acc1, acc2);
    grad_one_direction(B, M, xyz2, N, xyz1, graddist2, idx2, acc2, acc1);
    for (size_t t = 0; t < n1; t++) gradxyz1[t] = (float)acc1[t];
    for (size_t t = 0; t < n2; t++) gradxyz2[t] = (float)acc2[t];
    free(acc1);
    free(acc2);
}

/* ------------------------------------------------------------------------------------------------
 * EMD (auction) forward.  Follows emd_cuda_forward (emd_cuda.cu:228-282) and its kernels with the
 * initial state of emd_module.py:43-54 (assignment = assignment_inv = -1, price = 0,
 * max_increments = 0).  The reference's thread decomposition matters for exact ties and is
 * simulated literally:
 *   Bid (:95-179): block_cnt = n/256; unass_per_block = ceil(U/block_cnt); thread_per_unass =
 *     256/unass_per_block; inside each 2048-target chunk, thread t of a group scans the slice
 *     [t*delta, min((t+1)*delta, end_k)), delta = ceil(end_k/thread_per_unass) (:136-139); strict `>`
 *     in the scan (:147) and in the in-order group merge (:167).
 *     value = (float)((3.0 - (double)sqrtf(s)) - (double)price)   (:146, FP64 because of literal 3.0)
 *   calc_unass_idx (:85-93) compacts with atomicAdd -> order nondeterministic; the order only
 *     decides which block/group handles a point, never the result, so ascending order is used.
 *   GetMax (:181-194): every bidder within +-1e-6 (double) of the max writes max_idx, last writer
 *     wins -> racy in the reference.  ORACLE RULE: highest j wins (lowest j selectable, see the loop).
 *   Assign (:196-215) incl. the `last` iteration (no eviction, duplicates allowed).
 *   CalcDist (:217-226): dist = fma order of `deltax*deltax+deltay*deltay+deltaz*deltaz`,
 *     delta = xyz1 - xyz2.
 * Scratch arrays mirror the reference's caller-allocated tensors so state can be inspected.
 * Returns 1 on success, -1 on the shape violations of :236-249.
 * ---------------------------------------------------------------------------------------------- */
static int g_emd_getmax_lowest = 0;
void oracle_emd_set_getmax_rule(int lowest) { g_emd_getmax_lowest = lowest != 0; }

HOT int oracle_emd_forward(int B, int n, int m, const float *xyz1, const float *xyz2, float *dist,
                           int *assignment, float *price, int *assignment_inv, int *bid,
                           float *bid_increments, float *max_increments, int *unass_idx, int *max_idx,
                           float eps, int iters) {
    if (n != m) return -1;
    if (B > 512) return -1;
    if (n % 256 != 0) return -1;
    const int batch = 2048, block_size = 256, block_cnt = n / 256;
#pragma omp parallel for schedule(dynamic, 1)
    for (int i = 0; i < B; i++) {
        const float *p1 = xyz1 + (size_t)i * n * 3;
        const float *p2 = xyz2 + (size_t)i * n * 3;
        int *asg = assignment + (size_t)i * n;
        int *asg_inv = assignment_inv + (size_t)i * n;
        float *pr = price + (size_t)i * n;
        int *bd = bid + (size_t)i * n;
        float *binc = bid_increments + (size_t)i * n;
        float *minc = max_increments + (size_t)i * n;
        int *uidx = unass_idx + (size_t)i * n;
        int *midx = max_idx + (size_t)i * n;
        float tbest[256], tbetter[256];
        int tbest_i[256];
        for (int it = 0; it < iters; it++) {
            int last = (it == iters - 1);
            /* calc_unass_cnt / calc_unass_idx */
            int U = 0;
            for (int j = 0; j < n; j++)
                if (asg[j] == -1) uidx[U++] = j;
            if (U > 0) {
                /* Bid */
                int upb = (U + block_cnt - 1) / block_cnt;
                int tpu = block_size / upb;
                for (int u = 0; u < U; u++) {
                    int id = uidx[u];
                    float x1 = p1[id * 3 + 0], y1 = p1[id * 3 + 1], z1 = p1[id * 3 + 2];
                    for (int t = 0; t < tpu; t++) {
                        tbest[t] = -1e9f;
                        tbetter[t] = -1e9f;
                        tbest_i[t] = -1;
                    }
                    for (int k2 = 0; k2 < n; k2 += batch) {
                        int end_k = (n < k2 + batch ? n : k2 + batch) - k2;
                        int delta = (end_k + tpu - 1) / tpu;
                        for (int t = 0; t < tpu; t++) {
                            int l = t * delta;
                            int r = (t + 1) * delta < end_k ? (t + 1) * delta : end_k;
                            float best = tbest[t], better = tbetter[t];
                            int best_i = tbest_i[t];
                            for (int k = l; k < r; k++) {
                                int kk = k + k2;
                                float s = sqdist_ref(x1, y1, z1, p2[kk * 3 + 0], p2[kk * 3 + 1],
                                                     p2[kk * 3 + 2]);
                                float d = (float)((3.0 - (double)sqrtf(s)) - (double)pr[kk]);
                                if (d > best) {
                                    better = best;
                                    best = d;
                                    best_i = kk;
                                } else if (d > better) {
                                    better = d;
                                }
                            }
                            tbest[t] = best;
                            tbetter[t] = better;
                            tbest_i[t] = best_i;
                        }
                    }
                    float best = tbest[0], better = tbetter[0];
                    int best_i = tbest_i[0];
                    for (int t = 1; t < tpu; t++) {
                        if (tbest[t] > best) {
                            better = best > tbetter[t] ? best : tbetter[t];
                            best = tbest[t];
                            best_i = tbest_i[t];
                        } else {
                            better = better > tbest[t] ? better : tbest[t];
                        }
                    }
                    bd[id] = best_i;
                    float inc = best - better + eps;
                    binc[id] = inc;
                    if (inc > minc[best_i]) minc[best_i] = inc;
                }
            }
            /* GetMax: every bidder inside the +-1e-6 window stores its index, the last store wins (:188-191): a race with
             * no defined winner.  The oracle resolves it deterministically: HIGHEST j wins by default (the later thread /
             * block writes last -- what the reference did in every live comparison at n = 8192 / 16384 on B200), LOWEST j
             * when oracle_emd_set_getmax_rule(1) was called.  tests/golden/emd_ref_centered.npz is a witness of the race:
             * the reference's (run-to-run identical) output there equals the "lowest j" resolution and differs from the
             * "highest j" one in 44 of 1024 assignments; the other goldens have no decisive collision. */
            for (int jj = 0; jj < n; jj++) {
                const int j = g_emd_getmax_lowest ? n - 1 - jj : jj;
                if (asg[j] == -1) {
                    int bid_id = bd[j];
                    float bid_inc = binc[j];
                    float max_inc = minc[bid_id];
                    if ((double)bid_inc - 1e-6 <= (double)max_inc && (double)max_inc <= (double)bid_inc + 1e-6)
                        midx[bid_id] = j;
                }
            }
            /* Assign.  Evictions inside one launch are benign in the reference (an evicted point finds
             * max_idx[bid] != itself), so the decision is taken from the pre-launch `assignment`. */
            for (int u = 0; u < U; u++) {
                int j = uidx[u];
                int bid_id = bd[j];
                if (last || midx[bid_id] == j) {
                    float bid_inc = binc[j];
                    int ass_inv = asg_inv[bid_id];
                    if (!last && ass_inv != -1) asg[ass_inv] = -1;
                    asg_inv[bid_id] = j;
                    asg[j] = bid_id;
                    pr[bid_id] += bid_inc;
                    minc[bid_id] = -1e9f;
                }
            }
        }
        /* CalcDist */
        for (int j = 0; j < n; j++) {
            int k = asg[j];
            float dx = p1[j * 3 + 0] - p2[k * 3 + 0];
            float dy = p1[j * 3 + 1] - p2[k * 3 + 1];
            float dz = p1[j * 3 + 2] - p2[k * 3 + 2];
            dist[(size_t)i * n + j] = fmaf(dz, dz, fmaf(dx, dx, dy * dy));
        }
    }
    return 1;
}

/* EMD backward: NmDistanceGradKernel (emd_cuda.cu:284-300); gradient to xyz1 only, one term per
 * point so the atomicAdd onto zeros is exact: grad = 0 + g*(x1-x2). */
void oracle_emd_backward(int B, int n, const float *xyz1, const float *xyz2, const float *graddist,
                         const int *idx, float *gradxyz) {
    for (int i = 0; i < B; i++)
        for (int j = 0; j < n; j++) {
            size_t q = (size_t)i * n + j;
            int j2 = idx[q];
            size_t t = (size_t)i * n + j2;
            float g = graddist[q] * 2;
            gradxyz[q * 3 + 0] = 0.f + g * (xyz1[q * 3 + 0] - xyz2[t * 3 + 0]);
            gradxyz[q * 3 + 1] = 0.f + g * (xyz1[q * 3 + 1] - xyz2[t * 3 + 1]);
            gradxyz[q * 3 + 2] = 0.f + g * (xyz1[q * 3 + 2] - xyz2[t * 3 + 2]);
        }
}

/* ------------------------------------------------------------------------------------------------
 * Farthest point sampling.  The reference calls the un-vendored `fpsample.fps_sampling`
 * (main.py:21-22, reg_xyz.py:215, DepthPrompting.py:88) -> parity unpinned; semantics defined here:
 * start index given, running distance initialised to +inf, d = fma(dz,dz,fma(dx,dx,dy*dy)) with
 * d* = point - last_selected, running = min(running, d), next = argmax running, lowest index on ties.
 * Outputs idx[B,K] and (optionally) the selected running distance seq[B,K] (seq[.,0] = +inf).
 * ---------------------------------------------------------------------------------------------- */
HOT void oracle_fps(int B, int N, int K, int start, const float *xyz, int *idx, float *seq) {
#pragma omp parallel for schedule(dynamic, 1)
    for (int b = 0; b < B; b++) {
        const float *p = xyz + (size_t)b * N * 3;
        float *run = (float *)malloc(sizeof(float) * (N ? N : 1));
        for (int i = 0; i < N; i++) run[i] = INFINITY;
        int cur = start;
        for (int s = 0; s < K; s++) {
            idx[(size_t)b * K + s] = cur;
            float lx = p[cur * 3 + 0], ly = p[cur * 3 + 1], lz = p[cur * 3 + 2];
            float best = -1.f;
            int best_i = 0;
            for (int i = 0; i < N; i++) {
                float dx = p[i * 3 + 0] - lx, dy = p[i * 3 + 1] - ly, dz = p[i * 3 + 2] - lz;
                float d = fmaf(dz, dz, fmaf(dx, dx, dy * dy));
                float r = run[i] < d ? run[i] : d;
                run[i] = r;
                if (r > best) {
                    best = r;
                    best_i = i;
                }
            }
            if (seq && s == 0) seq[(size_t)b * K] = INFINITY;
            if (seq && s + 1 < K) seq[(size_t)b * K + s + 1] = best;
            cur = best_i;
        }
        free(run);
    }
}

/* ------------------------------------------------------------------------------------------------
 * Mean distance to the k nearest neighbours of every point of one cloud -- the per-point statistic of Open3D's
 * remove_statistical_outlier as the reference calls it on the fused cloud (reg_xyz.py:219, utils/dataUtils.py:652-666;
 * Open3D is not vendored: semantics restated from its documented behaviour, parity unpinned).  Squared distances with
 * the Chamfer rounding order, the k smallest kept, mean = (sum of their square roots, added in ascending order in
 * fp32) / count.  include_self counts the point itself (distance 0), as a KD-tree query of a cloud point does.
 * A cloud with fewer than k candidates averages what it has; none at all gives -1 (Open3D's marker).
 * ---------------------------------------------------------------------------------------------- */
HOT void oracle_knn_mean_distance(int n, int k, int include_self, const float *xyz, float *out) {
#pragma omp parallel for schedule(static)
    for (int i = 0; i < n; i++) {
        float best[32];
        for (int c = 0; c < k; c++) best[c] = INFINITY;
        const float qx = xyz[i * 3 + 0], qy = xyz[i * 3 + 1], qz = xyz[i * 3 + 2];
        for (int j = 0; j < n; j++) {
            if (!include_self && j == i) continue;
            float v = sqdist_ref(qx, qy, qz, xyz[j * 3 + 0], xyz[j * 3 + 1], xyz[j * 3 + 2]);
            if (!(v < best[k - 1])) continue;
            for (int c = 0; c < k; c++) { /* sorted insertion */
                const float lo = best[c] < v ? best[c] : v;
                v = best[c] < v ? v : best[c];
                best[c] = lo;
            }
        }
        float sum = 0.f;
        int m = 0;
        for (int c = 0; c < k; c++)
            if (best[c] < INFINITY) {
                sum = sum + sqrtf(best[c]);
                m++;
            }
        out[i] = m > 0 ? sum / (float)m : -1.0f;
    }
}

/* ------------------------------------------------------------------------------------------------
 * DepthPrompting geometry (DepthPrompting.py:239-271 getUvs, :179-184 pixel mapping, :292-391
 * paintPixels/getRawDepth).  Camera = 16 floats:
 *   [0..8]  R row-major (rows right / up / backward: camera looks down -z),  [9..11] t = -R*eye,
 *   [12] fx, [13] fy (= 1/tan(fovy/2), fx = fy/aspect), [14] A, [15] Bc   with z_ndc = A - Bc/depth
 *   (OpenGL projection with near/far: A = (far+near)/(far-near), Bc = 2*far*near/(far-near)).
 * kaolin is un-vendored -> parity unpinned; arithmetic defined here with explicit rounding:
 *   c = fma(R[.][2],pz, fma(R[.][1],py, fma(R[.][0],px, t[.])));  depth = -c_z
 *   ndc_x = (fx*c_x)/depth; ndc_y = (fy*c_y)/depth; ndc_z = A - Bc/depth
 * ---------------------------------------------------------------------------------------------- */
static inline void project_point(const float *cam, float px, float py, float pz, float *o) {
    float cx = fmaf(cam[2], pz, fmaf(cam[1], py, fmaf(cam[0], px, cam[9])));
    float cy = fmaf(cam[5], pz, fmaf(cam[4], py, fmaf(cam[3], px, cam[10])));
    float cz = fmaf(cam[8], pz, fmaf(cam[7], py, fmaf(cam[6], px, cam[11])));
    float depth = -cz;
    o[0] = (cam[12] * cx) / depth;
    o[1] = (cam[13] * cy) / depth;
    o[2] = cam[14] - cam[15] / depth;
}

/* getUvs: ndc[V,N,3], uv[V,N,2], bounds[V,4] = (cx, cy, scale, unused).  rescale as :247-262:
 * centre = (min+max)/2, scale = max(range_x, range_y), uv = ((xy-centre)/scale)*(1-2*padding)+0.5
 * (each step rounded separately; (1-2*padding) is formed in fp32 as 1.0f - 2.0f*padding).
 * rescale==0: uv = (xy+1)*0.5 (:264-266). */
void oracle_project_uv(int V, int N, const float *cams, const float *xyz, int rescale, float padding,
                       float *ndc, float *uv, float *bounds) {
    for (int v = 0; v < V; v++) {
        const float *cam = cams + v * 16;
        float mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
        for (int i = 0; i < N; i++) {
            float *o = ndc + ((size_t)v * N + i) * 3;
            project_point(cam, xyz[i * 3 + 0], xyz[i * 3 + 1], xyz[i * 3 + 2], o);
            mnx = fminf(mnx, o[0]);
            mxx = fmaxf(mxx, o[0]);
            mny = fminf(mny, o[1]);
            mxy = fmaxf(mxy, o[1]);
        }
        float cx = (mnx + mxx) / 2, cy = (mny + mxy) / 2;
        float rx = mxx - mnx, ry = mxy - mny;
        float sc = rx > ry ? rx : ry;
        float k = 1.0f - 2.0f * padding;
        if (bounds) {
            bounds[v * 4 + 0] = cx;
            bounds[v * 4 + 1] = cy;
            bounds[v * 4 + 2] = sc;
            bounds[v * 4 + 3] = k;
        }
        for (int i = 0; i < N; i++) {
            const float *o = ndc + ((size_t)v * N + i) * 3;
            float *w = uv + ((size_t)v * N + i) * 2;
            if (rescale) {
                w[0] = ((o[0] - cx) / sc) * k + 0.5f;
                w[1] = ((o[1] - cy) / sc) * k + 0.5f;
            } else {
                w[0] = (o[0] + 1.0f) * 0.5f;
                w[1] = (o[1] + 1.0f) * 0.5f;
            }
        }
    }
}

/* float -> unsigned key whose unsigned order equals the float order (handles negative ndc_z). */
static inline uint32_t float_order_key(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

/* z-buffer render.  Pixel mapping DepthPrompting.py:179-184: px = trunc(uv*res) (toward zero),
 * (row, col) = (px_v, px_u), clipped to [0,res-1]; splat the (2p-1)^2 square (:307-336) dropping
 * out-of-image taps; image flipped vertically at the end (:339) => stored row = res-1-row.
 * Where the reference lets an arbitrary point win a pixel (index_put, no depth test), the build
 * DEFINES: nearest ndc_z wins, ties -> lowest point index (packed (key<<32)|idx minimum).
 * Points with valid[i]==0 (if valid != NULL) are skipped.  zbuf[V,res,res] = packed word,
 * empty = 0xFFFFFFFFFFFFFFFF. */
void oracle_zbuffer(int V, int N, int res, int point_size, const float *uv, const float *ndc,
                    const unsigned char *valid, uint64_t *zbuf) {
    size_t npix = (size_t)V * res * res;
    for (size_t t = 0; t < npix; t++) zbuf[t] = ~(uint64_t)0;
    for (int v = 0; v < V; v++) {
        for (int i = 0; i < N; i++) {
            if (valid && !valid[(size_t)v * N + i]) continue;
            const float *w = uv + ((size_t)v * N + i) * 2;
            float z = ndc[((size_t)v * N + i) * 3 + 2];
            float fu = w[0] * (float)res, fv = w[1] * (float)res;
            if (!(fu == fu) || !(fv == fv) || !(z == z)) continue; /* NaN never paints */
            long col = (long)fu, row = (long)fv; /* trunc toward zero */
            if (fu >= 2147483647.0f) col = res - 1;
            if (fv >= 2147483647.0f) row = res - 1;
            if (fu <= -2147483648.0f) col = 0;
            if (fv <= -2147483648.0f) row = 0;
            if (col < 0) col = 0;
            if (col > res - 1) col = res - 1;
            if (row < 0) row = 0;
            if (row > res - 1) row = res - 1;
            uint64_t word = ((uint64_t)float_order_key(z) << 32) | (uint32_t)i;
            for (int dr = -point_size + 1; dr < point_size; dr++)
                for (int dc = -point_size + 1; dc < point_size; dc++) {
                    long r = row + dr, c = col + dc;
                    if (r < 0 || r >= res || c < 0 || c >= res) continue;
                    size_t o = ((size_t)v * res + (res - 1 - r)) * res + c;
                    if (word < zbuf[o]) zbuf[o] = word;
                }
        }
    }
}

/* Resolve a z-buffer: idx_img[V,res,res] (-1 empty), depth_img = 0.1+0.8*(1-(z-zmin)/(zmax-zmin))
 * (getRawDepth :362-366) over the points that own at least one pixel... the reference normalises
 * over the *visible input points*; here zmin/zmax are given per view by the caller. Empty = 0. */
void oracle_zbuffer_resolve(int V, int N, int res, const uint64_t *zbuf, const float *ndc,
                            const float *zminmax, int *idx_img, float *depth_img) {
    for (int v = 0; v < V; v++) {
        float zmin = zminmax[v * 2 + 0], zmax = zminmax[v * 2 + 1];
        float range = zmax - zmin;
        for (size_t p = 0; p < (size_t)res * res; p++) {
            uint64_t w = zbuf[(size_t)v * res * res + p];
            if (w == ~(uint64_t)0) {
                idx_img[(size_t)v * res * res + p] = -1;
                depth_img[(size_t)v * res * res + p] = 0.f;
            } else {
                int i = (int)(uint32_t)(w & 0xFFFFFFFFu);
                float z = ndc[((size_t)v * N + i) * 3 + 2];
                idx_img[(size_t)v * res * res + p] = i;
                depth_img[(size_t)v * res * res + p] = 0.1f + 0.8f * (1.0f - (z - zmin) / range);
            }
        }
    }
}

/* depth -> point unprojection (no reference counterpart; defined here).  For every non-empty pixel in
 * raster order (stored row r_s, col c): u = (c+0.5)/res, v = ((res-1-r_s)+0.5)/res (undo the flip),
 * ndc_xy = ((uv-0.5)/k)*scale + centre (inverse of the rescale), depth = Bc/(A - ndc_z) with ndc_z of
 * the owning point, cam = (ndc_x*depth/fx, ndc_y*depth/fy, -depth), world = R^T (cam - t) with
 * w_x = fma(R[2][0],d_z, fma(R[1][0],d_y, R[0][0]*d_x)) etc.  Output compacted out[V][count][3]
 * (capacity res*res per view), owner point index own[V][count], counts[V]. */
void oracle_unproject(int V, int N, int res, const float *cams, const float *bounds, int rescale,
                      const uint64_t *zbuf, const float *ndc, float *out, int *own, int *counts) {
    for (int v = 0; v < V; v++) {
        const float *cam = cams + v * 16;
        float cx = bounds[v * 4 + 0], cy = bounds[v * 4 + 1], sc = bounds[v * 4 + 2], k = bounds[v * 4 + 3];
        int cnt = 0;
        for (int rs = 0; rs < res; rs++)
            for (int c = 0; c < res; c++) {
                uint64_t w = zbuf[((size_t)v * res + rs) * res + c];
                if (w == ~(uint64_t)0) continue;
                int i = (int)(uint32_t)(w & 0xFFFFFFFFu);
                float z = ndc[((size_t)v * N + i) * 3 + 2];
                float u = ((float)c + 0.5f) / (float)res;
                float vv = ((float)(res - 1 - rs) + 0.5f) / (float)res;
                float nx, ny;
                if (rescale) {
                    nx = ((u - 0.5f) / k) * sc + cx;
                    ny = ((vv - 0.5f) / k) * sc + cy;
                } else {
                    nx = u * 2.0f - 1.0f;
                    ny = vv * 2.0f - 1.0f;
                }
                float depth = cam[15] / (cam[14] - z);
                float dx = (nx * depth) / cam[12] - cam[9];
                float dy = (ny * depth) / cam[13] - cam[10];
                float dz = -depth - cam[11];
                float *o = out + (((size_t)v * res * res) + cnt) * 3;
                o[0] = fmaf(cam[6], dz, fmaf(cam[3], dy, cam[0] * dx));
                o[1] = fmaf(cam[7], dz, fmaf(cam[4], dy, cam[1] * dx));
                o[2] = fmaf(cam[8], dz, fmaf(cam[5], dy, cam[2] * dx));
                own[(size_t)v * res * res + cnt] = i;
                cnt++;
            }
        counts[v] = cnt;
    }
}

/* ------------------------------------------------------------------------------------------------
 * Registration geometry (ObjectPoseOptim.forward, diff_obj_pose.py:408-436).
 * rotation_6d_to_matrix lives in un-vendored pytorch3d -> parity unpinned; restated from its published
 * definition (SURVEY.md appendix B): b1 = normalize(a1), b2 = normalize(a2 - (b1.a2) b1), b3 = b1 x b2,
 * rows of R; F.normalize = v / max(|v|, 1e-12).  Explicit rounding so the CUDA kernel can match bit for bit.
 * ---------------------------------------------------------------------------------------------- */
void oracle_pose_matrix(const float *d6, float *R) {
    float a1x = d6[0], a1y = d6[1], a1z = d6[2], a2x = d6[3], a2y = d6[4], a2z = d6[5];
    float n1 = fmaxf(sqrtf(fmaf(a1z, a1z, fmaf(a1y, a1y, a1x * a1x))), 1e-12f);
    float b1x = a1x / n1, b1y = a1y / n1, b1z = a1z / n1;
    float dp = fmaf(b1z, a2z, fmaf(b1y, a2y, b1x * a2x));
    float wx = a2x - dp * b1x, wy = a2y - dp * b1y, wz = a2z - dp * b1z;
    float n2 = fmaxf(sqrtf(fmaf(wz, wz, fmaf(wy, wy, wx * wx))), 1e-12f);
    float b2x = wx / n2, b2y = wy / n2, b2z = wz / n2;
    R[0] = b1x, R[1] = b1y, R[2] = b1z;
    R[3] = b2x, R[4] = b2y, R[5] = b2z;
    R[6] = b1y * b2z - b1z * b2y;
    R[7] = b1z * b2x - b1x * b2z;
    R[8] = b1x * b2y - b1y * b2x;
}

/* pts = R (s (V - c)) + c + t (diff_obj_pose.py:419-423), s = (float)exp((double)log_scale):
 * l = V - c; u = l*s; r_x = fma(R02,u_z, fma(R01,u_y, R00*u_x)); p_x = (r_x + c_x) + t_x. */
void oracle_transform(int N, const float *V, const float *c, const float *par, float *out) {
    float R[9];
    oracle_pose_matrix(par, R);
    float s = (float)exp((double)par[9]);
    for (int i = 0; i < N; i++) {
        float ux = (V[i * 3 + 0] - c[0]) * s, uy = (V[i * 3 + 1] - c[1]) * s, uz = (V[i * 3 + 2] - c[2]) * s;
        float rx = fmaf(R[2], uz, fmaf(R[1], uy, R[0] * ux));
        float ry = fmaf(R[5], uz, fmaf(R[4], uy, R[3] * ux));
        float rz = fmaf(R[8], uz, fmaf(R[7], uy, R[6] * ux));
        out[i * 3 + 0] = (rx + c[0]) + par[6];
        out[i * 3 + 1] = (ry + c[1]) + par[7];
        out[i * 3 + 2] = (rz + c[2]) + par[8];
    }
}

/* fp32 fused multiply-add, one rounding (C99 fmaf), elementwise over n values: out = a * b + c.  numpy has no fp32 fma and
 * float64 a * b + c rounds twice on the way to fp32, so tests that state a kernel's explicit fmaf order use this. */
void oracle_fmaf(int n, const float *a, const float *b, const float *c, float *out) {
    for (int i = 0; i < n; i++) out[i] = fmaf(a[i], b[i], c[i]);
}
