/*
 * genpc_b200.h -- C ABI of libgenpc_b200.so, the B200 (sm_100a) drop-in for GenPC's geometric hot path.
 *
 * Conventions (mirroring the reference's pybind surface, SURVEY.md section 8b):
 *   - every pointer is a DEVICE pointer unless the name starts with `h_` (host memory, pinned for full speed);
 *   - the caller owns every buffer, including outputs and workspaces; nothing is allocated or freed here
 *     (reference: dist_chamfer_3D.py:33-42, emd_module.py:43-54) -- the one exception is the genpc_host_feed_t
 *     handle, which owns a copy stream, two events and 260 B of flags;
 *   - clouds are contiguous AoS float[B][N][3] (chamfer3D.cu:19,23-25), indices are int32;
 *   - all work is enqueued on `stream` (a cudaStream_t; pass 0 for the legacy default stream the
 *     reference uses, chamfer3D.cu:142) and the call returns without synchronising;
 *   - return value: 0 = OK, >0 = cudaError_t of the failed launch, <0 = argument violation
 *     (GENPC_ERR_*).  The reference returns 1/0/-1 and prints (chamfer3D.cu:145-151,
 *     emd_cuda.cu:236-249); the Python mirrors translate.
 * There is no CPU fallback: without a CUDA device every entry point returns an error.
 */
#ifndef GENPC_B200_H
#define GENPC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void *genpc_stream_t; /* cudaStream_t */

#define GENPC_OK 0
#define GENPC_ERR_SHAPE (-1)     /* negative sizes, n != m, n % 256, B > 512 ... */
#define GENPC_ERR_WORKSPACE (-2) /* workspace NULL or too small */
#define GENPC_ERR_RANGE (-3)     /* B*N does not fit the 32-bit index space of the reference */

/* Experiment knobs (GENPC_* names, e.g. GENPC_FPS_MODE=cluster): the environment is read ONCE when the library is loaded;
 * genpc_set_tunable overrides a knob at run time (value NULL = unset), genpc_get_tunable returns the current value or NULL.
 * For tests and measurements; not synchronised with launches issued from other threads.  Unknown name: GENPC_ERR_SHAPE. */
int genpc_set_tunable(const char *name, const char *value);
const char *genpc_get_tunable(const char *name);

/* Library / build identification: returns a static string such as "genpc_b200 0.1 sm_100a". */
const char *genpc_version(void);

/* ---- Chamfer3D -------------------------------------------------------------------------------
 * Replaces chamfer_3D.forward (chamfer_cuda.cpp:17-19 -> chamfer_cuda_forward, chamfer3D.cu:136-154,
 * kernel NmDistanceKernel :12-134).
 *   dist1[b,j] = min_k |xyz1[b,j]-xyz2[b,k]|^2, idx1 = argmin (lowest k on ties); dist2/idx2 symmetric.
 *   Distance rounding is the reference's: fma(dz,dz,fma(dx,dx,dy*dy)).  Bit-exact outputs.
 * workspace: genpc_chamfer_workspace_bytes(B,N,M) bytes of device scratch (packed (dist,idx) words; for large cloud pairs --
 * at least 2^32 evaluations, more than 32768 points on one side, B <= 8 -- also the Hilbert-sorted copies, block boxes and
 * sort scratch of the pruned exact scan, csrc/nn_grid.cuh: same outputs bit for bit, 1M x 1M in 2.6 instead of 228 ms;
 * a workspace of only the packed words keeps such a call on the exhaustive kernels). */
size_t genpc_chamfer_workspace_bytes(int B, int N, int M);
int genpc_chamfer_forward(const float *xyz1, const float *xyz2, float *dist1, float *dist2, int *idx1,
                          int *idx2, int B, int N, int M, void *workspace, size_t workspace_bytes,
                          genpc_stream_t stream);

/* Diagnostics of the spatially pruned scan (GENPC_CHAMFER_PRUNE=1, csrc/nn_prune.cuh): launches add {target blocks fetched and
 * walked, query groups that needed the tie pass, query groups, 8-target chunks evaluated (the two-level scan of large clouds:
 * superblocks opened)} to the four device counters; NULL switches it off. */
int genpc_chamfer_prune_stats(unsigned *stats4);
/* Which scan genpc_chamfer_forward would queue for this shape with the current knobs (host logic only): 0 = exhaustive,
 * 1 = Hilbert-sorted pruned exact scan (batches of >= 2^30 evaluations, 2048 .. 32768 points per cloud), 2 = two-level pruned
 * exact scan for large clouds (>= 2^32 evaluations, more than 32768 points on a side, B <= 8).  Same outputs in every case. */
int genpc_chamfer_scan_kind(int B, int N, int M);
/* How the pruned scan's sort kernel would be laid out for B cloud pairs on a part with `sms` SMs (<= 0: 148; host logic only):
 * returns the CTAs per cloud of the larger side (1, or the thread-block cluster size 2 / 3 / 4 / 8), *mixed = 1 when the
 * smaller side's clouds take one CTA each, *grid = CTAs launched (whole clusters).  The rule keeps the grid inside one wave of
 * one 1024-thread CTA per SM; GENPC_SORT_CLUSTER overrides it. */
int genpc_chamfer_sort_layout(int B, int N, int M, int sms, int *mixed, int *grid);

/* Host-fed forward: the same result as genpc_chamfer_forward, but the clouds start in HOST memory
 * (h_xyz1 [B][N][3], h_xyz2 [B][M][3]; pinned memory for an asynchronous full-speed copy) and their transfer into the
 * caller's device buffers xyz1 / xyz2 is overlapped with the scan: the call cuts the batch into `chunks` groups of
 * cloud pairs (6 is a good value for a PCN batch: every chunk costs three copy-engine commands; clamped to [1, min(B, 64)]), copies them on the handle's private stream, and the ONE
 * scan launch on `stream` consumes each group as soon as its copy has landed.  This is the reference's stock flow
 * `xyz.cuda()` + chamfer_3D.forward (dist_chamfer_3D.py:33-47) with the 7 MB PCIe transfer of a PCN batch hidden
 * behind 0.27 ms of compute.  On return, all work is queued; `stream` is ordered after the copies, so xyz1 / xyz2 can
 * be used by later work on `stream` (e.g. genpc_chamfer_backward).  Batches large enough for the pruned exact scan (>= 2^30
 * distance evaluations, >= 2048 points per cloud) are cut in TWO chunks whatever `chunks` says, and each chunk's sort + scan
 * is queued on a stream of its own behind the chunk's copies instead of the one gated launch (same results; C2 forward from
 * pinned memory 0.33 -> 0.26 ms; GENPC_HOST_PRUNE=0 keeps the gated launch).  A handle serves one call at a time (host threads
 * sharing it are serialised by a lock inside the handle).  A gated launch that waits more than ~2 s for its data gives
 * up and raises the handle's error word: the fused form then returns loss = NaN, so the failure is seen at the first
 * natural synchronisation point; genpc_host_feed_error reports (synchronising `stream`) whether that happened since it
 * was last asked, and clears the word.
 * Every 256th call waits on the host for the previous call's copies (recycling of the pinned flag source ring). */
typedef struct genpc_host_feed genpc_host_feed_t;
int genpc_host_feed_create(genpc_host_feed_t **feed);
int genpc_host_feed_destroy(genpc_host_feed_t *feed);
int genpc_host_feed_inject_error(genpc_host_feed_t *feed, genpc_stream_t stream); /* test hook: raise the error word */
int genpc_host_feed_error(genpc_host_feed_t *feed, genpc_stream_t stream);
int genpc_chamfer_forward_host(genpc_host_feed_t *feed, const float *h_xyz1, const float *h_xyz2, float *xyz1,
                               float *xyz2, float *dist1, float *dist2, int *idx1, int *idx2, int B, int N, int M,
                               int chunks, void *workspace, size_t workspace_bytes, genpc_stream_t stream);

/* Fused forms of the two forward entries for a loss step (Completionloss.get_loss + backward, utils/loss_util.py:25-43
 * over dist_chamfer_3D.py:26-64): the ONE epilogue launch that follows the scan also
 *   - reduces the loss  loss_out[0] = w1 * mean f(dist1) + w2 * mean f(dist2)  (f = sqrt when use_sqrt; deterministic:
 *     one double partial per CTA, added in index order by the last CTA) -- what genpc_chamfer_loss does in its own launch;
 *   - zero-fills zero1 [B][N][3] / zero2 [B][M][3] (either may be NULL): the gradient accumulators that
 *     genpc_chamfer_backward / genpc_chamfer_loss_backward add into (dist_chamfer_3D.py:56-57 does it with two fills);
 *   - stores all-ones back into every packed word it consumed, so the NEXT fused call with the same B, N, M on the same
 *     `workspace` may pass workspace_armed = 1 and skip the memset.  (workspace_armed = 0 is always correct.)
 * A loss step is then 3 launches (scan, epilogue, gradient) instead of 7.  dist/idx outputs are unchanged, bit for bit.
 * loss_workspace: genpc_chamfer_fuse_workspace_bytes(B,N,M) bytes, zeroed ONCE by the caller (only read when loss_out
 * is not NULL).  fuse == NULL makes both calls identical to the plain entries.  Shapes that do not take the symmetric
 * path (tiny or empty clouds, GENPC_CHAMFER_MODE=scan) run the same duties as separate launches, re-arming included: after
 * any successful fused call with N > 0 and M > 0 the packed words are all-ones, whichever scan ran, and one loss workspace
 * serves calls of either path in any order. */
typedef struct genpc_chamfer_fuse {
    int workspace_armed;         /* in: the packed words of `workspace` are all-ones (left so by a previous fused call) */
    int use_sqrt;                /* loss: f = sqrt (chamfer_l1 forms) or identity (chamfer_l2 forms) */
    float w1, w2;                /* loss weights; a side with weight 0 is left out */
    float *loss_out;             /* device scalar, NULL: no loss */
    void *loss_workspace;
    size_t loss_workspace_bytes;
    float *zero1, *zero2;        /* device buffers to zero-fill, NULL: none */
} genpc_chamfer_fuse_t;
size_t genpc_chamfer_fuse_workspace_bytes(int B, int N, int M);
int genpc_chamfer_forward_fused(const float *xyz1, const float *xyz2, float *dist1, float *dist2, int *idx1, int *idx2,
                                int B, int N, int M, void *workspace, size_t workspace_bytes,
                                const genpc_chamfer_fuse_t *fuse, genpc_stream_t stream);
int genpc_chamfer_forward_host_fused(genpc_host_feed_t *feed, const float *h_xyz1, const float *h_xyz2, float *xyz1,
                                     float *xyz2, float *dist1, float *dist2, int *idx1, int *idx2, int B, int N, int M,
                                     int chunks, void *workspace, size_t workspace_bytes,
                                     const genpc_chamfer_fuse_t *fuse, genpc_stream_t stream);

/* Ragged batch: Chamfer distances (and, through `fuse`, the loss step) of cloud pairs of different sizes in one call.
 * len1 / len2 are device int32 [B] arrays, never NULL: pair b has len1[b] points at the start of its N-stride in xyz1 and
 * len2[b] at the start of its M-stride in xyz2; the device clamps them to [0, N] / [0, M] (0 is allowed).  Rows past a length
 * are never read (any value, NaN included).  For j < len1[b], dist1[b,j] / idx1[b,j] are bit for bit what
 * genpc_chamfer_forward returns for that pair alone on the sliced clouds (lowest index on ties); the same for dist2 / idx2.  A
 * row with no neighbour to report -- a padding row, or any row of a pair whose other cloud is empty -- gets dist 0 and idx -1,
 * so the gradient kernels give it zero gradient.  Fused loss: loss_out[0] = (1/B) sum_b [w1 mean_{j<len1[b]} f(dist1) +
 * w2 mean_{k<len2[b]} f(dist2)], a side with no points contributing 0 (lengths at the strides: the equal-size loss up to
 * summation order); zero-fill and re-arming as genpc_chamfer_forward_fused (every packed word, padding rows' included, so a fused
 * call leaves the workspace armed for the next call of either kind).  Workspaces: genpc_chamfer_workspace_bytes(B,N,M) and
 * genpc_chamfer_fuse_workspace_bytes(B,N,M).  A ragged call always runs the exhaustive symmetric scan, at every size: not the
 * per-direction scan of small clouds, nor the pruned scans (so a ragged batch of >= 2^30 evaluations with >= 2048 points per
 * cloud runs at the exhaustive rate, slower than an equal-size call), nor a host-fed launch.  GENPC_ERR_SHAPE for a NULL length
 * pointer or negative sizes, GENPC_ERR_WORKSPACE for a missing or too small workspace, GENPC_ERR_RANGE as the plain entry; all
 * before anything is queued.
 * genpc_chamfer_loss_backward_ragged is genpc_chamfer_loss_backward for the fused ragged loss: graddist = upstream[0] * w /
 * (B * len[b]) (* 0.5 / sqrt(dist) for f = sqrt); rows past a length contribute nothing.  The gradient of dist1 / dist2 of a
 * ragged forward goes through genpc_chamfer_backward unchanged (rows with idx -1 contribute nothing). */
int genpc_chamfer_forward_ragged(const float *xyz1, const float *xyz2, const int *len1, const int *len2, float *dist1,
                                 float *dist2, int *idx1, int *idx2, int B, int N, int M, void *workspace,
                                 size_t workspace_bytes, const genpc_chamfer_fuse_t *fuse /* NULL: plain forward */,
                                 genpc_stream_t stream);
int genpc_chamfer_loss_backward_ragged(const float *xyz1, const float *xyz2, const int *len1, const int *len2,
                                       const float *dist1, const float *dist2, const int *idx1, const int *idx2,
                                       const float *upstream, int use_sqrt, float w1, float w2, float *gradxyz1,
                                       float *gradxyz2, int B, int N, int M, genpc_stream_t stream);

/* Replaces chamfer_3D.backward (chamfer_cuda.cpp:22-27 -> chamfer_cuda_backward, chamfer3D.cu:176-195,
 * kernel NmDistanceGradKernel :155-174).  ACCUMULATES into gradxyz1/gradxyz2, which must arrive zeroed
 * exactly as in the reference (dist_chamfer_3D.py:56-57). */
int genpc_chamfer_backward(const float *xyz1, const float *xyz2, const float *graddist1,
                           const float *graddist2, const int *idx1, const int *idx2, float *gradxyz1,
                           float *gradxyz2, int B, int N, int M, genpc_stream_t stream);

/* Fused loss reductions over the forward outputs (the reference's Completionloss methods, utils/loss_util.py:25-43,
 * evaluate them with ~8 tiny torch launches per call and as many again in backward):
 *   out[0] = w1 * mean f(dist1) + w2 * mean f(dist2),  f = sqrt when use_sqrt (chamfer_l1: w1=w2=.5, chamfer_partial_l1:
 *   w1=1,w2=0) else identity (chamfer_l2: w1=w2=1, chamfer_partial_l2: w1=1,w2=0).  Deterministic single launch.
 * workspace: genpc_chamfer_loss_workspace_bytes() bytes, zeroed ONCE by the caller, reusable on the same stream.
 * genpc_chamfer_loss_backward accumulates d(loss)/d(xyz) * upstream[0] into gradxyz1/2 (zeroed by the caller), with the
 * per-point factor w/n (* 0.5/sqrt(dist)) folded into the six terms of NmDistanceGradKernel (chamfer3D.cu:155-174). */
size_t genpc_chamfer_loss_workspace_bytes(void);
int genpc_chamfer_loss(const float *dist1, const float *dist2, size_t n1, size_t n2, int use_sqrt, float w1, float w2,
                       float *out, void *workspace, size_t workspace_bytes, genpc_stream_t stream);
int genpc_chamfer_loss_backward(const float *xyz1, const float *xyz2, const float *dist1, const float *dist2,
                                const int *idx1, const int *idx2, const float *upstream, int use_sqrt, float w1, float w2,
                                float *gradxyz1, float *gradxyz2, int B, int N, int M, genpc_stream_t stream);

/* Target-sharded Chamfer (1M x 1M clouds over 2/4/8 GPUs; no reference counterpart -- the reference is
 * single-GPU brute force).  One direction against ONE shard of the targets: packed[b][j] =
 * min(packed[b][j], (dist_bits << 32) | (idx_base + k)).  Shards are merged by an all-reduce-MIN over the
 * 64-bit words (ncclInt64/ncclMin: the words are non-negative as int64 because dist >= 0; the low word makes
 * the lowest GLOBAL index win ties), then genpc_nn_unpack splits them into dist / idx.
 * init != 0 first fills packed with all-ones. */
int genpc_nn_partial_packed(const float *queries, const float *targets_shard, unsigned long long *packed, int B,
                            int Nq, int Mt_shard, int idx_base, int init, genpc_stream_t stream);
int genpc_nn_unpack(const unsigned long long *packed, float *dist, int *idx, size_t count, genpc_stream_t stream);

/* Row-sharded SYMMETRIC Chamfer: every point pair of the job is evaluated once.  Rank r scans its rows
 * [row_base, row_base+nr_shard) of cloud 1 (row_base % 128 == 0; B == 1 when row_base != 0) against ALL of cloud 2:
 * prow_shard[b][j] = final (dist, idx into cloud 2) of its rows, pcol[b][k] = min over its rows of
 * (dist, GLOBAL 128-row block id).  pcol is merged across ranks by all-reduce-MIN, then genpc_chamfer_sym_fixup
 * resolves each block id to the exact lowest row index against the FULL cloud 1 and writes dist/idx of cloud 2. */
int genpc_chamfer_sym_partial(const float *rows_shard, const float *cols, unsigned long long *prow_shard,
                              unsigned long long *pcol, int B, int nr_shard, int nc, int row_base, int init_cols,
                              genpc_stream_t stream);
int genpc_chamfer_sym_fixup(const float *rows_full, const float *cols, const unsigned long long *pcol, int B,
                            int nr_full, int nc, float *dist_cols, int *idx_cols, genpc_stream_t stream);

/* ---- k-NN statistic of the fusion tail ----------------------------------------------------------
 * Replaces the per-point part of Open3D's remove_statistical_outlier as the reference calls it on the fused cloud
 * (reg_xyz.py:219 -> utils/dataUtils.py:652-666, nb_neighbors=20; third-party CPU KD-tree code, not vendored):
 * mean_dist[i] = mean Euclidean distance from xyz[i] to its k nearest points of the same cloud (1 <= k <= 32);
 * include_self != 0 counts the point itself (distance 0) among the k, as a KD-tree query of a cloud point does.
 * Squared distances with the Chamfer rounding order, square roots added in ascending order in fp32: reproducible
 * bit for bit (oracle_knn_mean_distance).  A cloud with fewer than k candidates averages what it has; none: -1. */
int genpc_knn_mean_distance(const float *xyz, int n, int k, int include_self, float *mean_dist, genpc_stream_t stream);
/* Ragged batch: the same statistic for B clouds of different sizes in one launch.  xyz [B][n][3], mean_dist [B][n]; len is a
 * device int32 [B] array, never NULL: cloud b has len[b] points at the start of its n-stride, and the device clamps len[b] to
 * [0, n].  Rows past a length are never read (any value, NaN included).  For j < len[b], mean_dist[b][j] is bit for bit what
 * genpc_knn_mean_distance returns for that cloud alone on its len[b] points (include_self = 0 leaves out the query's own row of
 * its cloud); every row j in [len[b], n) gets -1, Open3D's marker of a query that found nothing.  n = 0 queues nothing.
 * GENPC_ERR_SHAPE, before anything is queued, for a NULL xyz, len or mean_dist, B outside [1, 65535] (the grid's y extent),
 * n < 0 and k outside [1, 32]. */
int genpc_knn_mean_distance_ragged(const float *xyz, const int *len, int B, int n, int k, int include_self,
                                   float *mean_dist, genpc_stream_t stream);

/* ---- surface sampling of the generated mesh -------------------------------------------------------
 * Replaces the sampling step of glb2point (utils/dataUtils.py:217-250: trimesh mesh.sample(num_points, return_index=True)
 * and the barycentric colour interpolation :231-243; third-party CPU code, unseeded), which turns the generated .glb
 * into the 163 840-point cloud reg() registers (reg_xyz.py:125) and the 120 000-point cloud of the differentiable init
 * (diff_obj_pose.py:504).  Semantics defined here (csrc/mesh.cu header, oracle/mesh.py): fp32 face areas without fma,
 * integer weights floor(area / max_area * 2^32) whose inclusive uint64 prefix sums the CALLER provides (exact, so the
 * face choice does not depend on summation order), counter-based splitmix64 draws from (seed, sample index).
 *   verts [n_verts][3] f32, faces [n_faces][3] i32, vertex_rgb [n_verts][3] f32 in [0,1] or NULL (-> 0.5 grey)
 *   areas [n_faces] f32 out (0 for degenerate / out-of-range faces)
 *   cum_weights [n_faces] u64 inclusive prefix sums, cum_weights[n_faces-1] > 0
 *   out_xyz [n_samples][3], out_rgb [n_samples][3] or NULL, out_face [n_samples] or NULL */
int genpc_mesh_face_areas(const float *verts, const int *faces, int n_verts, int n_faces, float *areas,
                          genpc_stream_t stream);
int genpc_mesh_sample(const float *verts, const int *faces, const float *vertex_rgb,
                      const unsigned long long *cum_weights, int n_faces, int n_samples, unsigned long long seed,
                      float *out_xyz, float *out_rgb, int *out_face, genpc_stream_t stream);

/* ---- point-to-point ICP step (scale / ICP candidate search) ----------------------------------------
 * Replaces one iteration of Open3D registration_icp(TransformationEstimationPointToPoint) as the reference calls it for
 * every scale candidate (reg_xyz.py:9-38 inside the sweeps :60-96 and :146-173; third-party CPU code), batched over K
 * candidates; the nearest neighbours come from genpc_chamfer_forward (dist1 / idx1 of cur vs target).
 *   cur [K][Ns][3]    the candidates' source clouds under their current transforms
 *   target [Kt][Nt][3], Kt = K or 1 (one target shared by all candidates)
 *   T [K][16]         row-major 4x4 transforms, updated in place: T <- [R|t] T, (R, t) = the least-squares rigid motion of
 *                     the inlier pairs (dist < max_dist2, NaN never, idx in [0, Nt)) -- Horn's closed form, identical
 *                     optimum to Kabsch/SVD; the sums are taken about the candidate's target row 0 (about the origin if
 *                     that row is not finite), so clouds far from the origin keep their precision
 *   state [K][4]      fitness, inlier_rmse, converged (0/1), calls -- zeroed by the caller before the first call; a
 *                     candidate converges when both |fitness - previous| < rel_fitness and |rmse - previous| < rel_rmse
 *                     (Open3D ICPConvergenceCriteria) and is left unchanged from then on, like one with < 3 inliers
 *   update = 0        statistics only (the evaluation after the last iteration)
 * One CTA per candidate, deterministic double accumulation, no host synchronisation. */
int genpc_icp_step(const float *cur, const float *target, const float *dist, const int *idx, float *T, float *state, int K,
                   int Ns, int Kt, int Nt, float max_dist2, float rel_fitness, float rel_rmse, int update,
                   genpc_stream_t stream);
/* Ragged batch: the same step for candidates of different sizes in one call.  src_len [K] / tgt_len [Kt] are device int32
 * arrays, never NULL: candidate k has src_len[k] points at the start of its Ns stride in source / cur and its target
 * tgt_len[k] (Kt = 1: tgt_len[0]) at the start of its Nt stride; the device clamps them to [0, Ns] / [0, Nt].  Rows past a
 * length are never read (any value, NaN included).  Inliers, fitness and rmse are taken over j < src_len[k] (fitness =
 * inliers / src_len[k]); an idx outside [0, tgt_len) is no inlier.  A candidate with 0 source or 0 target points has fitness 0
 * and rmse 0, never updates and gets no cur row written.
 *   source [K][Ns][3]  the untransformed clouds; after the step, cur[k][j] = T_k source[k][j] for j < src_len[k] (in place,
 *                      c_r = fma(T[r][2], z, fma(T[r][1], y, fma(T[r][0], x, T[r][3]))) in fp32): the next iteration's cur
 *   scan_len [K]       out: converged ? 0 : src_len[k] -- len1 of the next genpc_chamfer_forward_ragged, so that converged
 *                      candidates cost no scan work while the rest of the batch iterates
 * A candidate that enters a call converged reads no dist / idx (they are padding after scan_len = 0) and keeps T, fitness and
 * rmse; its calls counter still increments.  dist = idx = NULL: transform only (writes cur and scan_len, leaves T and state),
 * the call before a loop's first iteration.  Every candidate's T and state are bit for bit what it gets alone on its sliced
 * clouds.  GENPC_ERR_SHAPE, before anything is queued, for a NULL source or length pointer, only one of dist / idx NULL,
 * Kt not in {1, K} and sizes <= 0. */
int genpc_icp_step_ragged(const float *source, float *cur, const float *target, const float *dist, const int *idx,
                          const int *src_len, const int *tgt_len, int *scan_len, float *T, float *state, int K, int Ns,
                          int Kt, int Nt, float max_dist2, float rel_fitness, float rel_rmse, int update,
                          genpc_stream_t stream);

/* ---- Farthest point sampling -------------------------------------------------------------------
 * Replaces the reference's CPU call fpsample.fps_sampling(xyz, K) (main.py:21-22, reg_xyz.py:215,
 * DepthPrompting.py:88-90; un-vendored third-party package).  xyz [B][N][3] -> idx_out [B][K] int32,
 * first pick = `start`, lowest index on ties; seq_out (optional, may be NULL) [B][K] receives the running
 * distance of each pick (seq[.,0] = +inf; non-increasing afterwards).  One persistent CTA per cloud.
 * workspace: genpc_fps_workspace_bytes (0 unless N > 32768). */
size_t genpc_fps_workspace_bytes(int B, int N, int K);
int genpc_fps(const float *xyz, int B, int N, int K, int start, int *idx_out, float *seq_out,
              void *workspace, size_t workspace_bytes, genpc_stream_t stream);

/* ---- DepthPrompting geometry --------------------------------------------------------------------
 * Camera = 16 floats: [0..8] R row-major (rows right/up/backward), [9..11] t = -R*eye, [12] fx, [13] fy,
 * [14] A, [15] Bc with ndc_z = A - Bc/depth (OpenGL projection; kaolin semantics restated, DESIGN.md 3.4).
 *
 * genpc_project_uv replaces DepthPrompting.getUvs (DepthPrompting.py:239-271): cams[V][16], xyz[N][3] ->
 *   ndc[V][N][3] (the reference's `transformed_points`; ndc[..,2] is its `point_depths`), uv[V][N][2],
 *   bounds[V][4] = (centre_x, centre_y, scale, 1-2*padding) of the per-view rescale (may be NULL).
 * genpc_zbuffer_render replaces the pixel mapping (:179-184) + paintPixels/getRawDepth (:292-391):
 *   pixel = trunc(uv*res) -> (row=v, col=u), clipped, (2*point_size-1)^2 splat, vertical flip; a pixel is won
 *   by the nearest ndc_z, ties by the lowest point index (packed 64-bit atomicMin) -- where the reference's
 *   index_put lets an arbitrary point win.  valid[V][N] (uint8, may be NULL) masks points.
 *   Outputs (each may be NULL except zbuf): zbuf[V][res][res] packed words (empty = ~0), idx_img[V][res][res]
 *   (-1 empty), depth_img[V][res][res] = 0.1+0.8*(1-(z-zmin)/(zmax-zmin)) (0 empty), color_img[V][3][res][res]
 *   gathered from colors[N][3], zminmax[V][2].
 * genpc_unproject (no reference counterpart; defined in DESIGN.md 3.4): every non-empty pixel, in raster
 *   order, back to a 3-D point at the pixel centre: out[V][res*res][3], own[V][res*res], counts[V].
 * workspace for the first two: genpc_depth_workspace_bytes(V).  uv must be 8-byte aligned (it is accessed as float pairs;
 * GENPC_ERR_SHAPE otherwise); no other entry of this header needs more than the natural 4-byte alignment of its
 * arrays -- wider accesses are chosen at run time when the pointers allow them. */
size_t genpc_depth_workspace_bytes(int V);
int genpc_project_uv(const float *cams, const float *xyz, int V, int N, int rescale, float padding, float *ndc,
                     float *uv, float *bounds, void *workspace, size_t workspace_bytes, genpc_stream_t stream);
int genpc_zbuffer_render(const float *uv, const float *ndc, const unsigned char *valid, const float *colors,
                         int V, int N, int res, int point_size, unsigned long long *zbuf, int *idx_img,
                         float *depth_img, float *color_img, float *zminmax, void *workspace,
                         size_t workspace_bytes, genpc_stream_t stream);
int genpc_unproject(const float *cams, const float *bounds, int rescale, const unsigned long long *zbuf,
                    const float *ndc, int V, int N, int res, float *out, int *own, int *counts,
                    genpc_stream_t stream);

/* ---- EMD (auction) ------------------------------------------------------------------------------
 * Replaces emd.forward (emd.cpp:12-18 -> emd_cuda_forward, emd_cuda.cu:228-282; kernels clear :23,
 * calc_unass_cnt :30, calc_unass_cnt_sum :55, calc_unass_idx :85, Bid :95, GetMax :181, Assign :196,
 * CalcDist :217) with ONE persistent cooperative kernel.  Buffers and their required initial values are the
 * reference's (emd_module.py:43-54): assignment = assignment_inv = -1, price = bid_increments =
 * max_increments = 0; unass_cnt has >= B ints (the reference allocates 512).  The reference's
 * unass_cnt_sum / cnt_tmp scratch is not needed.  Returns GENPC_ERR_SHAPE for n != m, B > 512, n % 256 != 0
 * (emd_cuda.cu:236-249) and for eps <= 0 or iters <= 0 (the reference reads xyz2[-1] / mis-orders bids there).  Outputs dist[B][n], assignment[B][n] bit-identical to the reference wherever the
 * reference itself is deterministic (its GetMax store race is resolved as "highest bidder index"; the knob
 * GENPC_EMD_GETMAX=lowest -- environment at load time or genpc_set_tunable -- selects the other outcome the reference is
 * seen to produce).
 * workspace: genpc_emd_workspace_bytes_n(B, n) -- control words plus a spatially sorted copy of the targets (16 B per
 * target) and the boxes of its 64-target blocks, which let the Bid scan skip every block that cannot reach a bidder's
 * second-best value (bit-identical to the exhaustive scan; 64 <= n <= 32768).  A workspace of only
 * genpc_emd_workspace_bytes(B) bytes (control words only) is accepted and selects the exhaustive scan. */
size_t genpc_emd_workspace_bytes(int B);
size_t genpc_emd_workspace_bytes_n(int B, int n);
int genpc_emd_forward(const float *xyz1, const float *xyz2, float *dist, int *assignment, float *price,
                      int *assignment_inv, int *bid, float *bid_increments, float *max_increments,
                      int *unass_idx, int *unass_cnt, int *max_idx, int B, int n, int m, float eps, int iters,
                      void *workspace, size_t workspace_bytes, genpc_stream_t stream);
/* Replaces emd.backward (emd.cpp:20-23 -> emd_cuda_backward, emd_cuda.cu:302-316): gradient to xyz1 only,
 * ACCUMULATED into gradxyz (must arrive zeroed, emd_module.py:83). */
int genpc_emd_backward(const float *xyz1, const float *xyz2, float *gradxyz, const float *graddist,
                       const int *idx, int B, int n, genpc_stream_t stream);

/* ---- Fused registration loop (Geometric Preserving Fusion) --------------------------------------
 * Replaces the Chamfer part of the reference's pose/scale optimisation hot loop
 * (optim_registration/diff_obj_pose.py:518-576: ObjectPoseOptim.forward :408-436, Chamfer term of
 * compute_loss_function :323-334, loss.backward / Adam step / .item() :546-548) -- ONE kernel launch per
 * Adam iteration for all scans, no host synchronisation.
 *   complete[C][Nc][3]  moving clouds, center[C][3] their centroids, ref[C][Nr][3] fixed clouds, C = S/n_starts;
 *   scan i (one optimisation problem: a cloud pair x one multi-start) uses cloud pair i / n_starts;
 *   params[S][10] = rot_6d[6] | trans[3] | log_scale[1], adam_m / adam_v[S][10]: read and updated in place;
 *   loss_hist[S][T] (may be NULL): loss of iteration t written at column t, for t in [t_start, t_start+iters);
 *   loss = cd_weight * (w_fwd * mean sqrt NN(pts->ref) + w_inv * mean sqrt NN(ref->pts)), pts = R(s(V-c))+c+t;
 *   Adam betas (0.9, 0.999), eps 1e-8, step sizes lr_rot / lr_trans / lr_scale (diff_obj_pose.py:524-528).
 * workspace: genpc_register_workspace_bytes(S,Nc,Nr); pass reset_workspace=1 on the first call of a run
 * (later calls continuing the same run pass 0 and t_start = iterations already done). */
size_t genpc_register_workspace_bytes(int S, int Nc, int Nr);
/* Kernel launches per Adam iteration at this problem size: 1 (single fused launch) or 2 (symmetric scan + finish). */
int genpc_register_launches_per_iter(int S, int Nc, int Nr);
int genpc_register_run(const float *complete, const float *center, const float *ref, float *params,
                       float *adam_m, float *adam_v, float *loss_hist, int S, int n_starts, int Nc, int Nr,
                       int iters, int t_start, int T, double lr_rot, double lr_trans, double lr_scale,
                       float w_fwd, float w_inv, float cd_weight, void *workspace, size_t workspace_bytes,
                       int reset_workspace, genpc_stream_t stream);
/* Ragged batch: the same loop for cloud pairs of different sizes in one call.  Arguments are those of
 * genpc_register_run plus complete_len / ref_len (device int32 [C], never NULL): pair c has complete_len[c] moving
 * and ref_len[c] fixed points, stored at the start of its Nc / Nr stride; Nc / Nr are the padded strides and size
 * everything else (workspace: genpc_register_workspace_bytes(S,Nc,Nr)).  Each pair's loss is the mean over its own
 * points, so its trajectory is the one it has alone (up to the order of the partial sums); rows past a length are
 * never read (any value, NaN included).  Lengths are clamped to [1, Nc] / [1, Nr] on the device.  A ragged call always
 * runs one fused launch per iteration, at every size and whatever GENPC_REGISTER_MODE / GENPC_REGISTER_PERSIST say: the
 * persistent (all iterations in one launch), symmetric and pruned forms are not used, so a small ragged batch costs
 * the per-iteration launch chain and above S*Nc*Nr ~ 2e8 it is slower than an equal-size call.  Never synchronises; GENPC_ERR_SHAPE for a NULL
 * length pointer and for the shape errors of genpc_register_run. */
int genpc_register_run_ragged(const float *complete, const float *center, const float *ref, const int *complete_len,
                              const int *ref_len, float *params, float *adam_m, float *adam_v, float *loss_hist,
                              int S, int n_starts, int Nc, int Nr, int iters, int t_start, int T, double lr_rot,
                              double lr_trans, double lr_scale, float w_fwd, float w_inv, float cd_weight,
                              void *workspace, size_t workspace_bytes, int reset_workspace, genpc_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GENPC_B200_H */
