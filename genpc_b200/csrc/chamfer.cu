// chamfer.cu -- Chamfer3D nearest-neighbour forward / backward for sm_100a.
//
// Replaces the reference's NmDistanceKernel / NmDistanceGradKernel (chamfer3D.cu:12-195).
// Design (DESIGN.md section 4.1):
//   * one launch covers BOTH directions; a work item is (direction, batch, 256*QT queries, NN_SPAN targets),
//     so B=1 problems still fill 148 SMs (the reference runs 16 CTAs at B=1);
//   * targets are staged once per item into shared memory as SoA x[]/y[]/z[] (NaN padded), read back
//     with broadcast LDS.128, and evaluated two at a time on the packed FP32 pipe (FADD2/FMUL2/FFMA2);
//   * the running minimum is a single FMNMX3 per two pairs; the arg-min is NOT tracked per pair:
//     only the id of the 16-target chunk that lowered the minimum is kept (strict `<`, so the earliest
//     chunk wins ties) and the exact lowest index is recovered by re-scanning that one chunk;
//   * per-item results are merged across target splits with one packed 64-bit atomicMin per query
//     ((dist_bits << 32) | idx: unsigned order == dist ascending, then idx ascending == the reference's
//     lowest-index tie rule), then unpacked to dist/idx.
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>

#include "nn_core.cuh"
#include "nn_sym.cuh"
#include "nn_prune.cuh"
#include "nn_grid.cuh"

#ifndef GENPC_DEFAULT_SYM
#define GENPC_DEFAULT_SYM true
#endif
#ifndef GENPC_DEFAULT_BALANCED
#define GENPC_DEFAULT_BALANCED true
#endif

namespace genpc {

struct NNDir {
    const float *q;            // queries  [B][nq][3]
    const float *t;            // targets  [B][mt][3]
    unsigned long long *out;   // packed   [B][nq]
    int nq, mt, qtiles, tsplits, items;
    int idx_base;              // added to reported target indices (shard offset; 0 for plain Chamfer)
};
struct NNParams {
    NNDir dir[2];
};

template <int QT>
__global__ void __launch_bounds__(NN_THREADS, NN_MINBLOCKS) nn_scan_kernel(const NNParams p) {
    __shared__ __align__(16) float s[3][NN_SPAN];
    int item = blockIdx.x;
    const int d = (item >= p.dir[0].items) ? 1 : 0;
    if (d) item -= p.dir[0].items;
    // field-wise select keeps the parameters in constant memory (no local copy)
    const float *q = d ? p.dir[1].q : p.dir[0].q;
    const float *t = d ? p.dir[1].t : p.dir[0].t;
    unsigned long long *out = d ? p.dir[1].out : p.dir[0].out;
    const int nq = d ? p.dir[1].nq : p.dir[0].nq;
    const int mt = d ? p.dir[1].mt : p.dir[0].mt;
    const int qtiles = d ? p.dir[1].qtiles : p.dir[0].qtiles;
    const int tsplits = d ? p.dir[1].tsplits : p.dir[0].tsplits;
    const int idx_base = d ? p.dir[1].idx_base : p.dir[0].idx_base;
    const int ts = item % tsplits;
    const int rest = item / tsplits;
    const int qt = rest % qtiles;
    const int b = rest / qtiles;
    nn_scan_item<QT>(s, q + (size_t)b * nq * 3, nq, qt * (NN_THREADS * QT), t + (size_t)b * mt * 3, mt, ts * NN_SPAN,
                     idx_base, nullptr, nullptr, out + (size_t)b * nq);
}

// rearm: store all-ones back into every word after reading it, as the fused symmetric epilogue does (a fused call on the
// per-direction path leaves the workspace armed too)
__global__ void nn_unpack_kernel(unsigned long long *__restrict__ packed, float *__restrict__ dist1,
                                 int *__restrict__ idx1, size_t n1, float *__restrict__ dist2,
                                 int *__restrict__ idx2, size_t n2, int rearm) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n1 + n2) return;
    const unsigned long long w = packed[i];
    if (rearm) packed[i] = ~0ull;
    const float dv = __uint_as_float((unsigned int)(w >> 32));
    const int iv = (int)(unsigned int)(w & 0xffffffffu);
    if (i < n1) {
        dist1[i] = dv;
        idx1[i] = iv;
    } else {
        dist2[i - n1] = dv;
        idx2[i - n1] = iv;
    }
}

// += (x, y, z) on point `i` of an AoS [..][3] float array with TWO reductions instead of three: a point starts at byte
// 12*i, so either its (x, y) or its (y, z) pair is 8-byte aligned -- that pair goes out as one RED.ADD.F32x2, the
// remaining component as a scalar RED.  Addresses and operands are selected arithmetically (no divergence between the
// even and odd lanes of a warp).  VEC = false (array base not 8-byte aligned): three scalar reductions.
template <bool VEC>
__device__ __forceinline__ void red_add3(float *arr, size_t i, float x, float y, float z) {
    float *p = arr + i * 3;
    if (VEC) {
        const int odd = (int)(i & 1);
        atomicAdd(reinterpret_cast<float2 *>(p + odd), odd ? make_float2(y, z) : make_float2(x, y));
        atomicAdd(p + (odd ? 0 : 2), odd ? x : z);
    } else {
        atomicAdd(p, x);
        atomicAdd(p + 1, y);
        atomicAdd(p + 2, z);
    }
}

// Backward: same six terms as NmDistanceGradKernel (chamfer3D.cu:155-174): g = 2*grad; own += g*(p - nn); nn's -= g*(p - nn).
// GRAD_R points per thread, `nthreads` apart (coalesced): the chain idx -> gathered neighbour -> reductions is three dependent
// memory round trips per point, so every level is issued for all GRAD_R points before any is consumed (r02: one point per
// thread left the kernel latency bound at 0.17 of the HBM roofline).
constexpr int GRAD_R = 4;

// scatter term of one point, warp-aggregated: lanes that hit the same neighbour (common when many points of a dense cloud
// share one nearest neighbour in a sparse one and the cloud is stored with spatial locality) are summed by shuffles and issue
// ONE set of atomics.  Every lane of the warp must call this (invalid lanes carry unique keys).
template <bool VEC>
__device__ __forceinline__ void scatter_aggregated(float *go, bool valid, size_t t, int dir, float tx, float ty, float tz, int lane) {
    const unsigned long long key = valid ? ((unsigned long long)t * 2ull + (unsigned)dir) : (~0ull - (unsigned)lane);
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    if (peers == (1u << lane)) {
        if (valid) red_add3<VEC>(go, t, -tx, -ty, -tz);
        return;
    }
    const int leader = __ffs(peers) - 1;
    float sx = -tx, sy = -ty, sz = -tz;
    for (unsigned m = peers & (peers - 1u); m; m &= m - 1u) {  // every lane of the group runs the same trip count
        const int src = __ffs(m) - 1;
        const float ox = __shfl_sync(peers, -tx, src), oy = __shfl_sync(peers, -ty, src), oz = __shfl_sync(peers, -tz, src);
        sx += ox, sy += oy, sz += oz;
    }
    if (lane == leader) red_add3<VEC>(go, t, sx, sy, sz);  // groups only form among valid lanes
}

// LOSS = false: gd1 / gd2 are the upstream gradients of dist1 / dist2 (chamfer_3D.backward).
// LOSS = true : backward of the fused loss -- graddist = upstream[0] * w / n (* 0.5 / sqrt(d) for the L1 forms, inf at d == 0
//               exactly as torch's sqrt backward, loss_util.py:37); gd1 / gd2 are the forward's distances; w2 == 0 drops the
//               second direction.
// len1 / len2 (LOSS only; nullptr: full strides): points of each cloud of a ragged batch -- the mean of pair b's side runs over
// len[b] points, so graddist = upstream[0] * w / (B * len[b]); rows past a length and neighbours past the other cloud's length
// contribute nothing (genpc_chamfer_loss_backward_ragged).
template <bool VEC, bool LOSS>
__global__ void __launch_bounds__(256) chamfer_grad_kernel(const float *__restrict__ xyz1, const float *__restrict__ xyz2,
                                                          const float *__restrict__ gd1, const float *__restrict__ gd2,
                                                          const int *__restrict__ idx1, const int *__restrict__ idx2,
                                                          const float *__restrict__ upstream, int use_sqrt, float w1, float w2,
                                                          float *gx1, float *gx2, int B, int N, int M,
                                                          const int *__restrict__ len1 = nullptr,
                                                          const int *__restrict__ len2 = nullptr) {
    const size_t n1 = (size_t)B * N, n2 = (LOSS && w2 == 0.f) ? 0 : (size_t)B * M;
    const size_t nthreads = (size_t)gridDim.x * blockDim.x, g0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    bool valid[GRAD_R];
    int dir[GRAD_R], nn[GRAD_R];
    int lown[GRAD_R], loth[GRAD_R];   // ragged batch: points of the row's own cloud and of the other one
    size_t i[GRAD_R], t[GRAD_R];
    float x1[GRAD_R], y1[GRAD_R], z1[GRAD_R], gsc[GRAD_R], tx[GRAD_R], ty[GRAD_R], tz[GRAD_R];
    const float up = LOSS ? __ldg(upstream) : 0.f;
#pragma unroll
    for (int r = 0; r < GRAD_R; ++r) {   // level 1: index, own point, gradient scale
        i[r] = g0 + (size_t)r * nthreads;
        valid[r] = i[r] < n1 + n2;
        dir[r] = (valid[r] && i[r] >= n1) ? 1 : 0;
        if (dir[r]) i[r] -= n1;
        nn[r] = 0, x1[r] = y1[r] = z1[r] = gsc[r] = 0.f, lown[r] = loth[r] = 0;
        if (LOSS && len1 != nullptr && valid[r]) {   // ragged batch: a padding row is never read
            const int na = dir[r] ? M : N, b = (int)(i[r] / na);
            lown[r] = sym_len(dir[r] ? len2 : len1, b, na), loth[r] = sym_len(dir[r] ? len1 : len2, b, dir[r] ? N : M);
            valid[r] = (int)(i[r] - (size_t)b * na) < lown[r];
        }
        if (valid[r]) {
            const float *a = dir[r] ? xyz2 : xyz1;
            nn[r] = __ldg((dir[r] ? idx2 : idx1) + i[r]);
            x1[r] = __ldg(a + i[r] * 3), y1[r] = __ldg(a + i[r] * 3 + 1), z1[r] = __ldg(a + i[r] * 3 + 2);
            gsc[r] = __ldg((dir[r] ? gd2 : gd1) + i[r]);
        }
    }
#pragma unroll
    for (int r = 0; r < GRAD_R; ++r) {   // level 2: the gathered neighbour
        const int no = dir[r] ? N : M, na = dir[r] ? M : N;
        // an index outside [0, no) (caller-supplied garbage) contributes nothing instead of touching foreign memory
        valid[r] = valid[r] && (unsigned)nn[r] < (unsigned)no;
        if (LOSS && len1 != nullptr) valid[r] = valid[r] && nn[r] < loth[r];
        t[r] = 0, tx[r] = ty[r] = tz[r] = 0.f;
        if (valid[r]) {
            const float *o = dir[r] ? xyz1 : xyz2;
            t[r] = (i[r] / na) * no + nn[r];
            const float x2 = __ldg(o + t[r] * 3), y2 = __ldg(o + t[r] * 3 + 1), z2 = __ldg(o + t[r] * 3 + 2);
            float gd = gsc[r];
            if (LOSS) {
                const size_t cnt = len1 != nullptr ? (size_t)B * lown[r] : (dir[r] ? (size_t)B * M : n1);
                gd = __fmul_rn(up, __fdiv_rn(dir[r] ? w2 : w1, (float)cnt));
                if (use_sqrt) gd = __fmul_rn(gd, __fdiv_rn(0.5f, __fsqrt_rn(gsc[r])));
            }
            const float g = __fmul_rn(gd, 2.f);
            tx[r] = __fmul_rn(g, __fsub_rn(x1[r], x2));
            ty[r] = __fmul_rn(g, __fsub_rn(y1[r], y2));
            tz[r] = __fmul_rn(g, __fsub_rn(z1[r], z2));
        }
    }
#pragma unroll
    for (int r = 0; r < GRAD_R; ++r) {   // level 3: reductions
        // own term: one writer per element here, but the other direction scatters into the same array concurrently -> atomic
        if (valid[r]) red_add3<VEC>(dir[r] ? gx2 : gx1, i[r], tx[r], ty[r], tz[r]);
        scatter_aggregated<VEC>(dir[r] ? gx1 : gx2, valid[r], t[r], dir[r], tx[r], ty[r], tz[r], lane);
    }
}

static void fill_dir(NNDir &D, const float *q, const float *t, unsigned long long *out, int B, int nq, int mt,
                     int QT) {
    D.q = q, D.t = t, D.out = out, D.nq = nq, D.mt = mt;
    D.qtiles = (nq + NN_THREADS * QT - 1) / (NN_THREADS * QT);
    D.tsplits = (mt + NN_SPAN - 1) / NN_SPAN;
    D.items = B * D.qtiles * D.tsplits;
    D.idx_base = 0;
}

template <int QT>
static cudaError_t launch_scan(const NNParams &p, cudaStream_t stream) {
    const long long items = (long long)p.dir[0].items + p.dir[1].items;
    nn_scan_kernel<QT><<<(unsigned)items, NN_THREADS, 0, stream>>>(p);
    return cudaGetLastError();
}

// Spatially pruned exact scan (nn_prune.cuh, r02): Hilbert-ordered clouds, one warp per 32 queries, blocks visited nearest first.
// GENPC_CHAMFER_PRUNE=1 forces it for any shape it can take (64 .. 32768 points per cloud), =0 forbids it; by default it takes
// device-resident batches whose exhaustive scan is at least 2^30 distance evaluations with >= 2048 points per cloud -- BASELINE C2
// (32 x 2048 x 16384: forward 0.271 -> 0.196 ms), 32 x 8192 x 8192 (0.539 -> 0.292 ms); below that the fixed cost of the sort
// and of a group's dependent block chain (0.1 ms) loses (8 x 8192 x 8192: 0.155 vs 0.200 ms; profiles/r02m_chamfer_prune.txt).
// The first form (Z-order cells, a uniform global load per target) took 0.70 ms on C2.
static bool prune_shape_ok(int nr, int nc) { return nr >= PR_BLOCK && nc >= PR_BLOCK && nr <= PR_MAX_N && nc <= PR_MAX_N; }
static bool prune_eligible(int B, int nr, int nc) {
    if (!prune_shape_ok(nr, nc)) return false;
    const char *k = tunable("GENPC_CHAMFER_PRUNE");
    if (k != nullptr) return atoi(k) == 1;
    // (>= 2048 points per cloud: a thousand 1.8 K-point clouds -- the ICP scale search -- pay one sort CTA per cloud for next to
    // nothing: 72.6 vs 66.2 ms per search)
    return nr >= 2048 && nc >= 2048 && (long long)B * nr * nc >= (1LL << 30);
}
// Large clouds (nn_grid.cuh): multi-CTA sort + two-level pruned scan.  GENPC_CHAMFER_PRUNE=2 forces it for any shape it can
// take (and skips the probe below), =0 switches it off; by default it takes the shapes whose exhaustive scan is at least 2^32
// distance evaluations (>= 1 ms) with more than 32768 points on one side (BASELINE C5: 1M x 1M; not C1: 71 372 x 16 384).
static bool grid_shape_ok(int nr, int nc) { return nr >= PR_BLOCK && nc >= PR_BLOCK && nr <= GR_MAX_N && nc <= GR_MAX_N; }
static bool grid_eligible(int nr, int nc) {
    if (!grid_shape_ok(nr, nc)) return false;
    const char *k = tunable("GENPC_CHAMFER_PRUNE");
    if (k != nullptr) return atoi(k) == 2;
    return (long long)nr * nc >= (1LL << 32) && (nr > PR_MAX_N || nc > PR_MAX_N);
}
// The pruned scan of B cloud pairs (rows: the larger cloud) as genpc_chamfer_scan_kind reports it; the workspace size follows it
static int prune_kind(int B, int nr, int nc) { return B <= 8 && grid_eligible(nr, nc) ? 2 : (prune_eligible(B, nr, nc) ? 1 : 0); }
static void launch_prune2(const Prune2Params &q, cudaStream_t stream, bool probe) {
    const int groups = (q.nq + PR_GROUP - 1) / PR_GROUP;
    const int work = probe ? (groups + q.probe_stride - 1) / q.probe_stride : groups;
    const dim3 grid((unsigned)((work + PR_THREADS / 32 - 1) / (PR_THREADS / 32)), (unsigned)q.B);
    pr_rows(gr_nsb(q.nt), [&](auto r) {
        if (probe) nn_prune2_kernel<decltype(r)::value, true><<<grid, PR_THREADS, 0, stream>>>(q);
        else nn_prune2_kernel<decltype(r)::value, false><<<grid, PR_THREADS, 0, stream>>>(q);
    });
}
constexpr int GR_PROBE_GROUPS = 128;   // sampled query groups per direction and cloud

// The forward's workspace: the packed words (rows, then columns) and the control words of the pruned scans at its start -- a
// re-armed workspace is reused across calls -- then, from the next 256-byte boundary, the extras of pruned scan `kind`
struct ChamferWs {
    size_t bytes;
    int kind;
    unsigned long long *packed;   // [B][nr], then [B][nc]
    int *ctl;                     // [4]: [1] selection flag, [2] / [3] accumulator and ticket of the range check; [0] unused
    PruneSortParams prune;        // kind 1: sorted records, block and chunk boxes, every cloud's bounding box
    GridParams grid;              // kind 2: sorted records, block and superblock boxes, bounding box words, sort keys and values
    unsigned *keys_out;           //   ... and the radix sort's outputs (vals_out is grid.order) and scratch
    int *vals_out;
    void *cub_tmp;
    size_t cub_bytes;
};
static ChamferWs chamfer_layout(int B, int nr, int nc, int kind, void *base = nullptr) {
    WsCursor c{static_cast<char *>(base)};
    ChamferWs w = {};
    w.kind = kind, w.packed = c.take<unsigned long long>((size_t)B * nr + (size_t)B * nc);
    w.ctl = c.take<int>(4);
    const int n[2] = {nr, nc}, clouds[2] = {B, B};
    if (kind != 0) c.align_base();
    if (kind == 1) w.prune = pr_take_sorted(c, clouds, n), w.prune.bbx = c.take<float>((size_t)2 * B * 8);
    if (kind != 2) return w.bytes = c.bytes(), w;
    for (int i = 0; i < 2; ++i) {
        w.grid.sorted[i] = c.take<float4>((size_t)B * pr_npad(n[i]));
        w.grid.boxes[i] = c.take<float4>((size_t)B * 2 * pr_nblk(n[i]));
        w.grid.sboxes[i] = c.take<float4>((size_t)B * 2 * gr_nsb(n[i]));
    }
    for (int i = 0; i < 2; ++i) w.grid.bb[i] = c.take<int>((size_t)B * 8);
    // one cloud is sorted at a time: keys and values of the largest
    const int nmax = nr > nc ? nr : nc;
    w.grid.keys = c.take<unsigned>(nmax, 256), w.keys_out = c.take<unsigned>(nmax, 256);
    w.grid.vals = c.take<int>(nmax, 256), w.grid.order = w.vals_out = c.take<int>(nmax, 256);
    cub::DeviceRadixSort::SortPairs(nullptr, w.cub_bytes, (const unsigned *)nullptr, (unsigned *)nullptr, (const int *)nullptr,
                                    (int *)nullptr, nmax, 0, 30);
    w.cub_tmp = c.take<char>(w.cub_bytes, 256);
    return w.bytes = c.bytes(), w;
}

static unsigned *g_prune_stats = nullptr;   // diagnostics (genpc_chamfer_prune_stats), nullptr in production

// side stream + fork / join events for the cooperative kernel, one set per (device, caller stream): created on first use, kept
// for the life of the process (fork / join is also what a CUDA-graph capture of the step records)
struct PruneSide {
    cudaStream_t stream;
    cudaEvent_t fork, join;
};
static PruneSide *prune_side_stream(cudaStream_t caller) {
    static std::mutex mtx;
    static struct { int dev; cudaStream_t caller; PruneSide s; } tab[64];
    static int used = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> guard(mtx);
    for (int i = 0; i < used; ++i)
        if (tab[i].dev == dev && tab[i].caller == caller) return &tab[i].s;
    if (used == 64) return nullptr;   // (more caller streams than slots: the single-launch form)
    PruneSide s;
    if (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    tab[used].dev = dev, tab[used].caller = caller, tab[used].s = s;
    return &tab[used++].s;
}

static void launch_prune(const PruneParams &a, const PruneParams &b, cudaStream_t stream) {
    PrunePair pp = pr_pair(a, b);
    // few query groups against many target blocks (C2's partial -> complete direction): a CTA per group, eight warps sharing
    // its chain (nn_prune_coop_kernel) on a side stream, next to the other direction; GENPC_PRUNE_COOP=0 / 1 forbids / forces it
    const long long groups0 = (long long)pp.d[0].B * ((pp.d[0].nq + PR_GROUP - 1) / PR_GROUP);
    const char *ck = tunable("GENPC_PRUNE_COOP");
    const bool coop = ck != nullptr ? atoi(ck) != 0 : (groups0 <= 4096 && 4LL * pp.d[0].nq <= pp.d[1].nq);
    PruneSide *side = coop ? prune_side_stream(stream) : nullptr;
    if (side != nullptr) {
        cudaEventRecord(side->fork, stream);
        cudaStreamWaitEvent(side->stream, side->fork, 0);
        pr_rows(pr_nblk(pp.d[0].nt), [&](auto r) {
            nn_prune_coop_kernel<decltype(r)::value><<<(unsigned)groups0, PR_THREADS, 0, side->stream>>>(pp.d[0]);
        });
        cudaEventRecord(side->join, side->stream);
        pp.ctas0 = 0;   // the launch below: direction d[1] only
    }
    pr_launch(pp, stream);
    if (side != nullptr) cudaStreamWaitEvent(stream, side->join, 0);
}

// The sort of `clouds` clouds: one CTA per cloud, or a thread-block cluster of CS CTAs per cloud when one CTA per cloud would leave
// most SMs idle behind a few long CTAs (C2: 64 clouds, the 32 of 16384 points take 55 us in one CTA each).  GENPC_SORT_CLUSTER =
// 1 / 2 / 3 / 4 / 8 / m2 / m3 / m4 forces the layout (launch_bin_sort_cs: nn_prune.cuh).  Both sides of nb cloud pairs:
// The layout rule (host logic only; genpc_chamfer_sort_layout exposes it to the CPU tests): -> CTAs per cloud of the larger side,
// *mixed = 1 when the smaller side's clouds take one CTA each, *grid = CTAs launched.
static int sort_layout(int nb, int n0, int n1, int sms, int *mixed_out, int *grid_out) {
    const int nmax = n0 > n1 ? n0 : n1, nmin = n0 > n1 ? n1 : n0;
    int cs = 1, mixed = 0;
    const char *k = tunable("GENPC_SORT_CLUSTER");   // "2" / "3" / "4" / "8": every cloud a cluster; "m2" / "m3" / "m4": mixed layout
    if (k != nullptr) {
        mixed = k[0] == 'm' ? 1 : 0;
        cs = atoi(k + mixed);
        cs = cs >= 8 ? 8 : cs >= 4 ? 4 : cs == 3 ? 3 : cs == 2 ? 2 : 1;
    } else if (nmax >= 8192) {
        // as many CTAs per cloud as keep the grid inside one wave (one 1024-thread CTA per SM); when one side is much smaller, its
        // clouds take one CTA each and leave the SMs to the clusters of the larger side (C2: 32 x 3 + 33 CTAs)
        if (nmin * 4 <= nmax && nmin <= 4096) {
            mixed = 1;
            cs = nb * 4 + (nb + 3) / 4 * 4 <= sms ? 4 : nb * 3 + (nb + 2) / 3 * 3 <= sms ? 3 : nb * 2 + (nb + 1) / 2 * 2 <= sms ? 2 : 1;
        } else {
            cs = nb * 16 <= sms ? 8 : nb * 8 <= sms ? 4 : nb * 4 <= sms ? 2 : 1;
        }
    }
    if (cs < 2) mixed = 0;
    const int ctas = mixed ? nb * cs + nb : 2 * nb * cs;
    *mixed_out = mixed;
    *grid_out = (ctas + cs - 1) / cs * cs;
    return cs;
}

static void launch_bin_sort(PruneSortParams sp, int nb, cudaStream_t stream) {
    int mixed = 0, grid = 0;
    const int cs = sort_layout(nb, sp.n[0], sp.n[1], num_sms(), &mixed, &grid);
    sp.mixed = mixed;
    const int ctas = mixed ? nb * cs + nb : 2 * nb * cs;
    if (cs == 8) launch_bin_sort_cs<8>(sp, ctas, stream);
    else if (cs == 4) launch_bin_sort_cs<4>(sp, ctas, stream);
    else if (cs == 3) launch_bin_sort_cs<3>(sp, ctas, stream);
    else if (cs == 2) launch_bin_sort_cs<2>(sp, ctas, stream);
    else nn_bin_sort_kernel<1><<<2 * nb, PR_SORT_THREADS, 0, stream>>>(sp);
}

// Sort + pruned scan of the cloud pairs [b0, b0 + nb) of a batch of B (rows / cols: the batch's clouds; w: laid out for kind 1).
static int launch_prune_subbatch(const float *rows, const float *cols, int nr, int nc, const ChamferWs &w, int B, int b0, int nb,
                                 bool accumulate, cudaStream_t stream, int *chunk_ctl = nullptr) {
    PruneSortParams sp = w.prune;   // (the whole batch's buffers: advanced to pair b0 below)
    sp.xyz[0] = rows + (size_t)b0 * nr * 3, sp.xyz[1] = cols + (size_t)b0 * nc * 3, sp.B = nb;
    sp.limit = 1e15f, sp.ctl = chunk_ctl != nullptr ? chunk_ctl : w.ctl, sp.hilbert = 1, sp.accumulate = accumulate ? 1 : 0;
    sp.flag = chunk_ctl != nullptr ? w.ctl + 1 : nullptr;
    for (int i = 0; i < 2; ++i) {
        sp.sorted[i] += (size_t)b0 * pr_npad(sp.n[i]);
        sp.boxes[i] += (size_t)b0 * 2 * pr_nblk(sp.n[i]);
        sp.cboxes[i] += (size_t)b0 * 2 * (pr_npad(sp.n[i]) / 8);
    }
    sp.bbx += (size_t)b0 * 16;
    launch_bin_sort(sp, nb, stream);
    GENPC_CHECK_LAUNCH();
    PruneParams q = {};
    q.B = nb, q.select = w.ctl + 1, q.stats = g_prune_stats;
    q.q = sp.sorted[0], q.t = sp.sorted[1], q.tbox = sp.boxes[1], q.tcbox = sp.cboxes[1], q.out = w.packed + (size_t)b0 * nr, q.nq = nr,
    q.nt = nc;
    PruneParams q2 = q;
    q2.q = sp.sorted[1], q2.t = sp.sorted[0], q2.tbox = sp.boxes[0], q2.tcbox = sp.cboxes[0],
    q2.out = w.packed + (size_t)B * nr + (size_t)b0 * nc, q2.nq = nc, q2.nt = nr;
    launch_prune(q, q2, stream);
    GENPC_CHECK_LAUNCH();
    return GENPC_OK;
}

// The fused loss's workspace on the symmetric path: a double partial per epilogue CTA, then the ticket (in a 16-byte slot)
static size_t fuse_layout(int B, int N, int M, void *base, EpiFuse &f) {
    const size_t nr = (size_t)B * (N > M ? N : M), nc = (size_t)B * (N > M ? M : N);
    WsCursor c{static_cast<char *>(base)};
    f.partial = c.take<double>((nc + EPI_COLS_PER_CTA - 1) / EPI_COLS_PER_CTA + (nr + EPI_ROWS_PER_CTA - 1) / EPI_ROWS_PER_CTA);
    f.ticket = c.take<unsigned>(4);
    return c.bytes();
}

// Symmetric path: rows = the larger cloud (registers), cols = the smaller one (shared-memory sweep).
// gate != nullptr: host-fed launch (nn_sym_gated_kernel), see genpc_chamfer_forward_host.
// len1 / len2 != nullptr: ragged batch (genpc_chamfer_forward_ragged; w laid out for kind 0, no gate).
static int chamfer_forward_sym(const float *xyz1, const float *xyz2, float *dist1, float *dist2, int *idx1, int *idx2,
                               int B, int N, int M, const ChamferWs &w, cudaStream_t stream,
                               const unsigned *gate = nullptr, unsigned gate_gen = 0, int gate_pairs = 1,
                               const genpc_chamfer_fuse_t *fuse = nullptr, const int *prune_chunks = nullptr,
                               const int *len1 = nullptr, const int *len2 = nullptr) {
    const bool swap = M > N;
    SymParams p = {};
    p.rows = swap ? xyz2 : xyz1, p.cols = swap ? xyz1 : xyz2;
    p.nr = swap ? M : N, p.nc = swap ? N : M;
    p.len_r = swap ? len2 : len1, p.len_c = swap ? len1 : len2;
    float *dist_r = swap ? dist2 : dist1, *dist_c = swap ? dist1 : dist2;
    int *idx_r = swap ? idx2 : idx1, *idx_c = swap ? idx1 : idx2;
    p.prow = w.packed, p.pcol = w.packed + (size_t)B * p.nr;
    p.rblock_base = 0;
    p.gate = gate, p.gate_gen = gate_gen, p.gate_pairs = gate_pairs;
    p.select = nullptr;
    // ---- spatially pruned scan of w.kind (0: none; the workspace holds its extras): both it and the exhaustive kernel below are
    // queued; the selection flag ctl[1], written by the sort's range check or by the grid probe, decides on the device which one
    // does the work.  ctl[2] / ctl[3]: accumulator and ticket of the range check (ctl[2] also counts the probe's block visits) ----
    int *ctl = w.ctl;
    const bool use_grid = w.kind == 2, use_prune = w.kind != 0;
    if (use_grid) {
        GridParams gp = w.grid;
        gp.B = B, gp.limit = 1e15f, gp.ctl = ctl;
        gp.xyz[0] = p.rows, gp.xyz[1] = p.cols, gp.n[0] = p.nr, gp.n[1] = p.nc;
        const int nmax = p.nr > p.nc ? p.nr : p.nc;
        size_t cub_bytes = w.cub_bytes;
        int ctas = (nmax + 4095) / 4096;
        if (ctas > 4 * GENPC_NUM_SMS) ctas = 4 * GENPC_NUM_SMS;
        if (ctas < 1) ctas = 1;
        grid_init_kernel<<<1, 256, 0, stream>>>(gp);
        grid_bbox_kernel<<<dim3(ctas, B, 2), GR_THREADS, 0, stream>>>(gp);
        GENPC_CHECK_LAUNCH();
        for (int side = 0; side < 2; ++side)
            for (int b = 0; b < B; ++b) {   // (large clouds come in small batches)
                grid_key_kernel<<<ctas, GR_THREADS, 0, stream>>>(gp, side, b);
                cudaError_t es = cub::DeviceRadixSort::SortPairs(w.cub_tmp, cub_bytes, (const unsigned *)gp.keys, w.keys_out,
                                                                 (const int *)gp.vals, w.vals_out, gp.n[side], 0, 30, stream);
                if (es != cudaSuccess) return (int)es;
                grid_gather_kernel<<<ctas, GR_THREADS, 0, stream>>>(gp, side, b, side == 0 && b == 0);
            }
        GENPC_CHECK_LAUNCH();
        const int nblk_max = pr_nblk(nmax), nsb_max = gr_nsb(nmax);
        grid_boxes_kernel<false><<<dim3((nblk_max + 7) / 8, B, 2), GR_THREADS, 0, stream>>>(gp);
        grid_boxes_kernel<true><<<dim3((nsb_max + 7) / 8, B, 2), GR_THREADS, 0, stream>>>(gp);
        GENPC_CHECK_LAUNCH();
        p.select = ctl + 1;
        Prune2Params q = {};
        q.B = B, q.select = ctl + 1, q.stats = g_prune_stats;
        // data-dependent guard: a sample of the query groups runs first and counts its block visits; when a group needs more
        // than a tenth of the target blocks on average (clouds that do not overlap, e.g. BASELINE C1's scan against an
        // unrelated shape) the exhaustive kernels are faster and take over through the selection flag
        const char *pk = tunable("GENPC_CHAMFER_PRUNE");
        const bool forced = pk != nullptr && atoi(pk) == 2;
        for (int pass = forced ? 1 : 0; pass < 2; ++pass) {
            const bool probe = pass == 0;
            long long limit = 0;
            for (int dir = 0; dir < 2; ++dir) {
                q.q = gp.sorted[dir], q.t = gp.sorted[1 - dir], q.tbox = gp.boxes[1 - dir], q.tsbox = gp.sboxes[1 - dir];
                q.out = dir == 0 ? p.prow : p.pcol, q.nq = gp.n[dir], q.nt = gp.n[1 - dir];
                const int groups = (q.nq + PR_GROUP - 1) / PR_GROUP, nblk = pr_nblk(q.nt);
                q.probe_stride = groups > GR_PROBE_GROUPS ? groups / GR_PROBE_GROUPS : 1;
                q.probe_cap = nblk / 5 > 64 ? nblk / 5 : 64;
                q.probe_acc = ctl + 2;
                const long long sampled = (long long)B * ((groups + q.probe_stride - 1) / q.probe_stride);
                limit += sampled * (nblk / 10 > 16 ? nblk / 10 : 16);
                launch_prune2(q, stream, probe);
            }
            if (probe) grid_decide_kernel<<<1, 1, 0, stream>>>(ctl, (int)(limit > 0x7fffffffLL ? 0x7fffffffLL : limit));
        }
        GENPC_CHECK_LAUNCH();
    } else if (use_prune) {
        if (prune_chunks == nullptr) {
            const int rcp = launch_prune_subbatch(p.rows, p.cols, p.nr, p.nc, w, B, 0, B, false, stream);
            if (rcp != GENPC_OK) return rcp;
        } else {
            // the caller (host-fed batches) has already queued sort + scan chunk by chunk as the copies landed; a LATER chunk may
            // have asked for the exhaustive kernels after earlier ones stored exact words: start those over
            prune_rearm_kernel<<<2 * GENPC_NUM_SMS, 256, 0, stream>>>(p.prow, (size_t)B * (p.nr + p.nc), ctl + 1);
            GENPC_CHECK_LAUNCH();
        }
        p.select = ctl + 1;
    }
    // measured on B200 (profiles/r01c_sym_variants.txt): QT=4 at 3 CTAs/SM is within 1 % of QT=8 at 2 CTAs/SM on
    // large clouds and clearly better when the grid is small
    const int QT = p.nr >= 1024 ? 4 : 2;
    const long long items = sym_tiling(B, p.nr, p.nc, QT, p.rtiles, p.span, p.cspans);
    if (items > 0x7fffffffLL) return GENPC_ERR_RANGE;
    // measured on B200 (profiles/r01h_sym_balanced_vs_grid.txt): with fewer than two waves of full-span work items the
    // balanced form wins (B=1 16384^2 +5 %, 3 x 5000 x 3333 +12 %); with more, one CTA per item is 4-5 % faster (resident
    // CTAs drift out of phase, so staging / publishing of one overlaps the scan of the other)
    const char *bm = tunable("GENPC_SYM_BALANCED");
    const bool few_items = (long long)B * p.rtiles * ((p.nc + SYM_SPAN_MAX - 1) / SYM_SPAN_MAX) < 4LL * GENPC_NUM_SMS;
    // Behind a pruned scan this launch is only the device-selected fall-back, and a fixed-size grid returns at once: one CTA per
    // work item of a 1M x 1M pair spent 0.8 ms launching CTAs that do nothing (grid scan), and C2's 2048 items were a 3-4 us
    // launch between the pruned scan and the epilogue.  When the fall-back does run (out-of-range, far-apart or collapsed clouds)
    // C2-sized batches pay the balanced form's 4-5 % (above) -- inputs already off the fast path.  Behind the Hilbert-sorted
    // pruned scan it is also a programmatic dependent (launch_pdl): of nn_prune_kernel, or of the join with the cooperative kernel
    // A ragged batch always takes the item grid (nn_sym_kernel): the balanced form has no per-cloud lengths (SymParams)
    const bool balanced = p.len_r == nullptr &&
                          ((bm == nullptr) ? ((GENPC_DEFAULT_BALANCED && few_items) || use_prune) : (atoi(bm) != 0));
    const bool dep = w.kind == 1;
    cudaError_t es = cudaSuccess;
    if (gate != nullptr) {
        if (QT >= 4) nn_sym_gated_kernel<4><<<(unsigned)items, SYM_THREADS, 0, stream>>>(p);
        else nn_sym_gated_kernel<2><<<(unsigned)items, SYM_THREADS, 0, stream>>>(p);
    } else if (balanced) {
        // balanced grid: 2 resident CTAs per SM, each walks an equal share of the (row tile x 32-column block) units
        const int upj = (p.nc + 31) / 32;
        const long long units = (long long)B * p.rtiles * upj;
        if (units > 0x7fffffffLL) return GENPC_ERR_RANGE;
        const int grid = (int)(units < 2LL * GENPC_NUM_SMS ? units : 2LL * GENPC_NUM_SMS);
        auto kb = QT == 4 ? nn_sym_balanced_kernel<4> : nn_sym_balanced_kernel<2>;
        if (dep) es = launch_pdl(kb, dim3(grid), dim3(SYM_THREADS), stream, p, (int)units, upj);
        else kb<<<grid, SYM_THREADS, 0, stream>>>(p, (int)units, upj);
    } else {
        auto kg = QT == 4 ? nn_sym_kernel<4> : nn_sym_kernel<2>;
        if (dep) es = launch_pdl(kg, dim3((unsigned)items), dim3(SYM_THREADS), stream, p);
        else kg<<<(unsigned)items, SYM_THREADS, 0, stream>>>(p);
    }
    if (es != cudaSuccess) return (int)es;
    GENPC_CHECK_LAUNCH();
    const size_t nrw = (size_t)B * p.nr, ncw = (size_t)B * p.nc;
    const unsigned fix_blocks = (unsigned)((ncw + EPI_COLS_PER_CTA - 1) / EPI_COLS_PER_CTA);
    const unsigned unpack_blocks = (unsigned)((nrw + EPI_ROWS_PER_CTA - 1) / EPI_ROWS_PER_CTA);
    EpiFuse f;
    memset(&f, 0, sizeof(f));
    // column words are exact iff the pruned scan did the work (ctl[1] == 0)
    f.select = use_prune ? ctl + 1 : nullptr;
    f.len_r = p.len_r, f.len_c = p.len_c;
    // the epilogue is a programmatic dependent of the scan launched above (whichever it is: every one of them triggers early)
    const dim3 egrid(fix_blocks + unpack_blocks);
    if (fuse == nullptr) {
        es = launch_pdl(nn_sym_epilogue_kernel<false>, egrid, dim3(256), stream, p.rows, p.cols, p.prow, p.pcol, B, p.nr, p.nc, 32 * QT,
                        fix_blocks, dist_r, idx_r, dist_c, idx_c, f);
    } else {
        // dist1 belongs to xyz1: the row cloud unless the clouds were swapped; a ragged batch divides each term by its pair's
        // length in the epilogue, the 1 / B here
        const bool ragged = len1 != nullptr;
        const double f1 = (fuse->w1 != 0.f) ? (double)fuse->w1 / (double)(ragged ? (size_t)B : (size_t)B * N) : 0.0;
        const double f2 = (fuse->w2 != 0.f) ? (double)fuse->w2 / (double)(ragged ? (size_t)B : (size_t)B * M) : 0.0;
        f.frow = swap ? f2 : f1, f.fcol = swap ? f1 : f2;
        f.use_sqrt = fuse->use_sqrt, f.rearm = 1;
        if (fuse->loss_out != nullptr) fuse_layout(B, N, M, fuse->loss_workspace, f), f.loss_out = fuse->loss_out;
        f.zero[0] = fuse->zero1, f.nzero[0] = (size_t)B * N * 3;
        f.zero[1] = fuse->zero2, f.nzero[1] = (size_t)B * M * 3;
        f.err_flag = gate != nullptr ? gate + GATE_ERR_SLOT : nullptr;
        es = launch_pdl(nn_sym_epilogue_kernel<true>, egrid, dim3(256), stream, p.rows, p.cols, p.prow, p.pcol, B, p.nr, p.nc, 32 * QT,
                        fix_blocks, dist_r, idx_r, dist_c, idx_c, f);
    }
    if (es != cudaSuccess) return (int)es;
    return GENPC_OK;
}

}  // namespace genpc

using namespace genpc;

extern "C" size_t genpc_chamfer_workspace_bytes(int B, int N, int M) {
    if (B < 0 || N < 0 || M < 0) return 0;
    const int nr = N > M ? N : M, nc = N > M ? M : N;
    return chamfer_layout(B, nr, nc, prune_kind(B, nr, nc)).bytes;
}

static bool takes_sym_path(int N, int M) {
    // "sym": one evaluation of every distance feeds both directions (nn_sym.cuh); "scan": one scan per direction
    const char *mode = tunable("GENPC_CHAMFER_MODE");
    const bool want_sym = (mode == nullptr) ? GENPC_DEFAULT_SYM : (strcmp(mode, "sym") == 0);
    return want_sym && N > 0 && M > 0 && (N > M ? N : M) >= 512;
}

// The loss workspace holds the fused epilogue's partials and ticket, then, from the next 16-byte boundary, those of the plain loss
// kernel (the per-direction path).  Each kernel zeroes only its own ticket, so the two must not overlap: one workspace serves
// calls of either path in any order (GENPC_CHAMFER_MODE flipped between calls of one shape).
static size_t plain_loss_offset(int B, int N, int M) {
    EpiFuse f;
    return (fuse_layout(B, N, M, nullptr, f) + 15) & ~(size_t)15;
}

extern "C" size_t genpc_chamfer_fuse_workspace_bytes(int B, int N, int M) {
    if (B < 0 || N < 0 || M < 0) return 0;
    return plain_loss_offset(B, N, M) + genpc_chamfer_loss_workspace_bytes();
}

// The unfused tail of a fused call, for the shapes that do not take the symmetric path (tiny or empty clouds).
static int fuse_tail_unfused(const genpc_chamfer_fuse_t *fuse, const float *dist1, const float *dist2, int B, int N, int M,
                             cudaStream_t stream) {
    cudaError_t e;
    const size_t n1 = (size_t)B * N, n2 = (size_t)B * M;
    if (fuse->zero1 != nullptr && n1) {
        e = cudaMemsetAsync(fuse->zero1, 0, n1 * 12, stream);
        if (e != cudaSuccess) return (int)e;
    }
    if (fuse->zero2 != nullptr && n2) {
        e = cudaMemsetAsync(fuse->zero2, 0, n2 * 12, stream);
        if (e != cudaSuccess) return (int)e;
    }
    if (fuse->loss_out == nullptr) return GENPC_OK;
    const size_t off = plain_loss_offset(B, N, M);
    return genpc_chamfer_loss(dist1, dist2, n1, n2, fuse->use_sqrt, fuse->w1, fuse->w2, fuse->loss_out,
                              static_cast<char *>(fuse->loss_workspace) + off, fuse->loss_workspace_bytes - off,
                              (genpc_stream_t)stream);
}

static int fuse_check(const genpc_chamfer_fuse_t *fuse, int B, int N, int M) {
    if (fuse == nullptr || fuse->loss_out == nullptr) return GENPC_OK;
    if (fuse->loss_workspace == nullptr || fuse->loss_workspace_bytes < genpc_chamfer_fuse_workspace_bytes(B, N, M))
        return GENPC_ERR_WORKSPACE;
    return GENPC_OK;
}

extern "C" int genpc_chamfer_forward_fused(const float *xyz1, const float *xyz2, float *dist1, float *dist2,
                                           int *idx1, int *idx2, int B, int N, int M, void *workspace,
                                           size_t workspace_bytes, const genpc_chamfer_fuse_t *fuse,
                                           genpc_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (B < 0 || N < 0 || M < 0) return GENPC_ERR_SHAPE;
    int rc = fuse_check(fuse, B, N, M);
    if (rc != GENPC_OK) return rc;
    const size_t n1 = (size_t)B * N, n2 = (size_t)B * M;
    if (n1 + n2 == 0) return fuse ? fuse_tail_unfused(fuse, dist1, dist2, B, N, M, stream) : GENPC_OK;
    if (N == 0 || M == 0) {
        // the reference's kernels write nothing in this case; outputs keep the zeros they were allocated with
        if (n1) {
            cudaMemsetAsync(dist1, 0, n1 * 4, stream);
            cudaMemsetAsync(idx1, 0, n1 * 4, stream);
        }
        if (n2) {
            cudaMemsetAsync(dist2, 0, n2 * 4, stream);
            cudaMemsetAsync(idx2, 0, n2 * 4, stream);
        }
        GENPC_CHECK_LAUNCH();
        return fuse ? fuse_tail_unfused(fuse, dist1, dist2, B, N, M, stream) : GENPC_OK;
    }
    const int nr = N > M ? N : M, nc = N > M ? M : N;
    if (workspace == nullptr || workspace_bytes < chamfer_layout(B, nr, nc, 0).bytes) return GENPC_ERR_WORKSPACE;
    const bool sym = takes_sym_path(N, M);
    // (a workspace sized while the knob was off stays on the exhaustive kernels)
    int kind = sym ? prune_kind(B, nr, nc) : 0;
    if (workspace_bytes < chamfer_layout(B, nr, nc, kind).bytes) kind = 0;
    const ChamferWs w = chamfer_layout(B, nr, nc, kind, workspace);
    cudaError_t e;
    // an armed workspace already holds all-ones words: a fused call on either path leaves them so
    if (!(fuse != nullptr && fuse->workspace_armed)) {
        e = cudaMemsetAsync(w.packed, 0xff, (n1 + n2) * 8, stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(w.ctl, 0, 16, stream);
        if (e != cudaSuccess) return (int)e;
    }
    if (sym) return chamfer_forward_sym(xyz1, xyz2, dist1, dist2, idx1, idx2, B, N, M, w, stream, nullptr, 0, 1, fuse);

    const int QT = nn_pick_qt(N < M ? N : M);
    NNParams p;
    fill_dir(p.dir[0], xyz1, xyz2, w.packed, B, N, M, QT);
    fill_dir(p.dir[1], xyz2, xyz1, w.packed + n1, B, M, N, QT);
    const long long items = (long long)p.dir[0].items + p.dir[1].items;
    if (items > 0x7fffffffLL) return GENPC_ERR_RANGE;
    switch (QT) {
        case 4: nn_scan_kernel<4><<<(unsigned)items, NN_THREADS, 0, stream>>>(p); break;
        case 2: nn_scan_kernel<2><<<(unsigned)items, NN_THREADS, 0, stream>>>(p); break;
        default: nn_scan_kernel<1><<<(unsigned)items, NN_THREADS, 0, stream>>>(p); break;
    }
    GENPC_CHECK_LAUNCH();
    const size_t tot = n1 + n2;
    nn_unpack_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, stream>>>(w.packed, dist1, idx1, n1, dist2, idx2, n2,
                                                                        fuse != nullptr ? 1 : 0);
    GENPC_CHECK_LAUNCH();
    return fuse ? fuse_tail_unfused(fuse, dist1, dist2, B, N, M, stream) : GENPC_OK;
}

extern "C" int genpc_chamfer_forward(const float *xyz1, const float *xyz2, float *dist1, float *dist2,
                                     int *idx1, int *idx2, int B, int N, int M, void *workspace,
                                     size_t workspace_bytes, genpc_stream_t stream_) {
    return genpc_chamfer_forward_fused(xyz1, xyz2, dist1, dist2, idx1, idx2, B, N, M, workspace, workspace_bytes, nullptr,
                                       stream_);
}

// Ragged batch: pair b has len1[b] / len2[b] points at the start of its N / M stride (clamped to [0, stride] on the device); rows
// past a length are never read and get dist 0 / idx -1, like every row of a pair whose other cloud is empty.  Always the
// exhaustive symmetric scan, at every size: the per-direction, pruned, grid and host-fed scans have no per-cloud counts.
extern "C" int genpc_chamfer_forward_ragged(const float *xyz1, const float *xyz2, const int *len1, const int *len2, float *dist1,
                                            float *dist2, int *idx1, int *idx2, int B, int N, int M, void *workspace,
                                            size_t workspace_bytes, const genpc_chamfer_fuse_t *fuse, genpc_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (len1 == nullptr || len2 == nullptr || B < 0 || N < 0 || M < 0) return GENPC_ERR_SHAPE;
    int rc = fuse_check(fuse, B, N, M);
    if (rc != GENPC_OK) return rc;
    const size_t n1 = (size_t)B * N, n2 = (size_t)B * M;
    cudaError_t e = cudaSuccess;
    if (n1 == 0 || n2 == 0) {
        // every pair has an empty side: no row has a neighbour, and the loss (a mean of zeros, or of nothing) is 0
        if (n1 && e == cudaSuccess) e = cudaMemsetAsync(dist1, 0, n1 * 4, stream);
        if (n1 && e == cudaSuccess) e = cudaMemsetAsync(idx1, 0xff, n1 * 4, stream);
        if (n2 && e == cudaSuccess) e = cudaMemsetAsync(dist2, 0, n2 * 4, stream);
        if (n2 && e == cudaSuccess) e = cudaMemsetAsync(idx2, 0xff, n2 * 4, stream);
        if (e != cudaSuccess) return (int)e;
        return fuse ? fuse_tail_unfused(fuse, dist1, dist2, B, N, M, stream) : GENPC_OK;
    }
    const int nr = N > M ? N : M, nc = N > M ? M : N;
    if (workspace == nullptr || workspace_bytes < chamfer_layout(B, nr, nc, 0).bytes) return GENPC_ERR_WORKSPACE;
    // chamfer_forward_sym's range check of its item grid, before anything is queued
    int rtiles = 0, span = 0, cspans = 0;
    if (sym_tiling(B, nr, nc, nr >= 1024 ? 4 : 2, rtiles, span, cspans) > 0x7fffffffLL) return GENPC_ERR_RANGE;
    const ChamferWs w = chamfer_layout(B, nr, nc, 0, workspace);
    if (!(fuse != nullptr && fuse->workspace_armed)) {  // (the fused epilogue re-arms every word, padding rows' included)
        e = cudaMemsetAsync(w.packed, 0xff, (n1 + n2) * 8, stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(w.ctl, 0, 16, stream);
        if (e != cudaSuccess) return (int)e;
    }
    return chamfer_forward_sym(xyz1, xyz2, dist1, dist2, idx1, idx2, B, N, M, w, stream, nullptr, 0, 1, fuse, nullptr, len1, len2);
}

extern "C" int genpc_chamfer_backward(const float *xyz1, const float *xyz2, const float *graddist1,
                                      const float *graddist2, const int *idx1, const int *idx2,
                                      float *gradxyz1, float *gradxyz2, int B, int N, int M,
                                      genpc_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (B < 0 || N < 0 || M < 0) return GENPC_ERR_SHAPE;
    const size_t tot = (size_t)B * N + (size_t)B * M;
    if (tot == 0 || N == 0 || M == 0) return GENPC_OK;
    // vector reductions need 8-byte aligned gradient arrays (every point then has one aligned component pair)
    const bool vec = ((reinterpret_cast<size_t>(gradxyz1) | reinterpret_cast<size_t>(gradxyz2)) & 7) == 0;
    const unsigned grid = (unsigned)((tot + 256 * GRAD_R - 1) / (256 * GRAD_R));
    if (vec)
        chamfer_grad_kernel<true, false><<<grid, 256, 0, stream>>>(xyz1, xyz2, graddist1, graddist2, idx1, idx2, nullptr, 0, 0.f, 0.f,
                                                                  gradxyz1, gradxyz2, B, N, M);
    else
        chamfer_grad_kernel<false, false><<<grid, 256, 0, stream>>>(xyz1, xyz2, graddist1, graddist2, idx1, idx2, nullptr, 0, 0.f, 0.f,
                                                                   gradxyz1, gradxyz2, B, N, M);
    GENPC_CHECK_LAUNCH();
    return GENPC_OK;
}

// The pruned scan's sort layout for B cloud pairs on a part with `sms` SMs (<= 0: 148) -- sort_layout above, host logic only.
extern "C" int genpc_chamfer_sort_layout(int B, int N, int M, int sms, int *mixed, int *grid) {
    if (B <= 0 || N <= 0 || M <= 0 || mixed == nullptr || grid == nullptr) return GENPC_ERR_SHAPE;
    return sort_layout(B, N > M ? N : M, N > M ? M : N, sms > 0 ? sms : GENPC_NUM_SMS_B200, mixed, grid);
}

// Which scan genpc_chamfer_forward would queue for this shape with the current knobs (host logic only, no device call):
// 0 = exhaustive (symmetric or per-direction), 1 = Hilbert-sorted pruned scan (nn_prune.cuh), 2 = two-level pruned scan for large
// clouds (nn_grid.cuh).  The device may still hand a pruned launch back to the exhaustive kernels (range / overlap / probe).
extern "C" int genpc_chamfer_scan_kind(int B, int N, int M) {
    if (B <= 0 || N <= 0 || M <= 0) return GENPC_ERR_SHAPE;
    if (!takes_sym_path(N, M)) return 0;
    return prune_kind(B, N > M ? N : M, N > M ? M : N);
}

// diagnostics of the pruned scan: stats4 = device pointer to 4 counters (blocks walked, groups that took the tie pass, groups,
// 8-target chunks evaluated; nn_grid.cuh: superblocks opened)
extern "C" int genpc_chamfer_prune_stats(unsigned *stats4) {
    g_prune_stats = stats4;
    return GENPC_OK;
}

extern "C" const char *genpc_version(void) { return "genpc_b200 0.1 sm_100a"; }

// ---- host-fed Chamfer forward: the H2D copy of the clouds overlaps the scan ------------------------------------------
// The e2e form of the hot call (BASELINE metric measured from HOST buffers): the clouds are cut into `chunks` groups of
// cloud pairs; a private copy stream moves chunk after chunk from (pinned) host memory into the caller's device
// buffers and, behind every chunk, DMA-writes the call's generation number into that chunk's gate word.  ONE full-size
// nn_sym_gated_kernel is launched right after the first chunk has been queued: its CTAs run in batch order and only
// wait when they get ahead of the copy engine (PCIe: 7 MB = 0.13 ms for C2, the scan: 0.27 ms), so the transfer costs
// one chunk of latency instead of the whole copy.  Flags are written by the copy engine, never by a kernel or memset
// (those need SM resources the resident scan CTAs hold).
struct genpc_host_feed {
    cudaStream_t copy_stream;
    cudaEvent_t ready, copied;
    cudaEvent_t chunk_ev[GATE_MAX_CHUNKS];   // chunked pruned path: chunk c's copies have landed
    cudaEvent_t done_ev[GATE_MAX_CHUNKS];    //   ... its sort + scan have finished
    cudaEvent_t fork;
    cudaStream_t cstream[GATE_MAX_CHUNKS];   //   ... the stream they run on (chunks overlap each other and the copies)
    int *cctl;                               //   ... per-chunk accumulator / ticket words of the sort kernel (device, zero between launches)
    unsigned *gate;    // device: GATE_MAX_CHUNKS generation words + the error word
    unsigned *h_ring;  // pinned: source words of the gate writes
    unsigned gen;
    int device;
    std::mutex lock;   // one call at a time per handle: the generation counter, the ring slot and the gate words are shared
};
static constexpr int FEED_RING = 256;

extern "C" int genpc_host_feed_create(genpc_host_feed_t **out) {
    if (out == nullptr) return GENPC_ERR_SHAPE;
    genpc_host_feed *f = new (std::nothrow) genpc_host_feed();
    if (f == nullptr) return (int)cudaErrorMemoryAllocation;
    f->copy_stream = nullptr, f->ready = nullptr, f->copied = nullptr, f->gate = nullptr, f->h_ring = nullptr, f->gen = 0;
    for (int c = 0; c < GATE_MAX_CHUNKS; ++c) f->chunk_ev[c] = nullptr, f->done_ev[c] = nullptr, f->cstream[c] = nullptr;
    f->fork = nullptr, f->cctl = nullptr;
    cudaError_t e = cudaGetDevice(&f->device);
    for (int c = 0; c < GATE_MAX_CHUNKS && e == cudaSuccess; ++c) {
        e = cudaEventCreateWithFlags(&f->chunk_ev[c], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&f->done_ev[c], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&f->fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc((void **)&f->cctl, GATE_MAX_CHUNKS * 4 * sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(f->cctl, 0, GATE_MAX_CHUNKS * 4 * sizeof(int));
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&f->copy_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&f->ready, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&f->copied, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc((void **)&f->gate, (GATE_MAX_CHUNKS + 1) * sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMemset(f->gate, 0, (GATE_MAX_CHUNKS + 1) * sizeof(unsigned));
    if (e == cudaSuccess) e = cudaHostAlloc((void **)&f->h_ring, FEED_RING * sizeof(unsigned), cudaHostAllocDefault);
    if (e != cudaSuccess) {
        genpc_host_feed_destroy(f);
        return (int)e;
    }
    *out = f;
    return GENPC_OK;
}

extern "C" int genpc_host_feed_destroy(genpc_host_feed_t *f) {
    if (f == nullptr) return GENPC_OK;
    if (f->copy_stream) cudaStreamSynchronize(f->copy_stream), cudaStreamDestroy(f->copy_stream);
    if (f->ready) cudaEventDestroy(f->ready);
    if (f->copied) cudaEventDestroy(f->copied);
    for (int c = 0; c < GATE_MAX_CHUNKS; ++c) {
        if (f->chunk_ev[c]) cudaEventDestroy(f->chunk_ev[c]);
        if (f->done_ev[c]) cudaEventDestroy(f->done_ev[c]);
        if (f->cstream[c]) cudaStreamSynchronize(f->cstream[c]), cudaStreamDestroy(f->cstream[c]);
    }
    if (f->fork) cudaEventDestroy(f->fork);
    if (f->cctl) cudaFree(f->cctl);
    if (f->gate) cudaFree(f->gate);
    if (f->h_ring) cudaFreeHost(f->h_ring);
    delete f;
    return GENPC_OK;
}

extern "C" int genpc_chamfer_forward_host(genpc_host_feed_t *f, const float *h_xyz1, const float *h_xyz2, float *xyz1,
                                          float *xyz2, float *dist1, float *dist2, int *idx1, int *idx2, int B, int N,
                                          int M, int chunks, void *workspace, size_t workspace_bytes,
                                          genpc_stream_t stream_) {
    return genpc_chamfer_forward_host_fused(f, h_xyz1, h_xyz2, xyz1, xyz2, dist1, dist2, idx1, idx2, B, N, M, chunks, workspace,
                                            workspace_bytes, nullptr, stream_);
}

extern "C" int genpc_chamfer_forward_host_fused(genpc_host_feed_t *f, const float *h_xyz1, const float *h_xyz2, float *xyz1,
                                                float *xyz2, float *dist1, float *dist2, int *idx1, int *idx2, int B,
                                                int N, int M, int chunks, void *workspace, size_t workspace_bytes,
                                                const genpc_chamfer_fuse_t *fuse, genpc_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (f == nullptr || B < 0 || N < 0 || M < 0) return GENPC_ERR_SHAPE;
    const size_t n1 = (size_t)B * N, n2 = (size_t)B * M;
    if (n1 + n2 == 0)
        return genpc_chamfer_forward_fused(xyz1, xyz2, dist1, dist2, idx1, idx2, B, N, M, workspace, workspace_bytes, fuse, stream_);
    const int frc = fuse_check(fuse, B, N, M);
    if (frc != GENPC_OK) return frc;
    cudaError_t e;
#define FEED_CHECK(x) do { e = (x); if (e != cudaSuccess) return (int)e; } while (0)
    const bool sym = takes_sym_path(N, M);
    if (!sym || B < 2 || chunks < 2) {
        // tiny clouds / a single pair: nothing worth overlapping -- copy on the caller's stream, then the plain entry
        if (n1) FEED_CHECK(cudaMemcpyAsync(xyz1, h_xyz1, n1 * 12, cudaMemcpyHostToDevice, stream));
        if (n2) FEED_CHECK(cudaMemcpyAsync(xyz2, h_xyz2, n2 * 12, cudaMemcpyHostToDevice, stream));
        return genpc_chamfer_forward_fused(xyz1, xyz2, dist1, dist2, idx1, idx2, B, N, M, workspace, workspace_bytes, fuse, stream_);
    }
    const int nr_ = M > N ? M : N, nc_ = M > N ? N : M;
    if (workspace == nullptr || workspace_bytes < chamfer_layout(B, nr_, nc_, 0).bytes) return GENPC_ERR_WORKSPACE;
    std::lock_guard<std::mutex> guard(f->lock);   // host threads sharing the handle take turns (ADVICE r01)
    if (chunks > GATE_MAX_CHUNKS) chunks = GATE_MAX_CHUNKS;
    if (chunks > B) chunks = B;
    const int pairs = (B + chunks - 1) / chunks;  // cloud pairs per chunk
    chunks = (B + pairs - 1) / pairs;
    // ---- pruned scan (the default for batches of this size): sort + scan are queued per chunk behind an event of the chunk's
    // copies -- no kernel waits on a gate, the last chunk's sort + scan (a few tens of us) is all that follows the last copy ----
    // MEASURED r02 (C2 forward from pinned memory, same box, tools/time_hostfeed.py -> profiles/r02w_time_hostfeed.json): gated
    // exhaustive launch 0.326-0.334 ms (6 / 8 chunks), this path 0.260-0.270 ms (2-6 chunks, one stream per chunk; all chunks on the
    // caller's stream: 0.81 ms, each chunk's sort + scan bound by its own latency).  Before the sort kernel spread a cloud over a
    // cluster a chunk of five clouds was five 55-us CTAs and the two paths tied (0.371 vs 0.361 ms per step) -- default since then;
    // GENPC_HOST_PRUNE=0 keeps the gated launch.
    const char *hp = tunable("GENPC_HOST_PRUNE");
    if ((hp == nullptr || atoi(hp) == 1) && prune_kind(B, nr_, nc_) == 1 && workspace_bytes >= chamfer_layout(B, nr_, nc_, 1).bytes) {
        const ChamferWs w = chamfer_layout(B, nr_, nc_, 1, workspace);
        const float *rows = M > N ? xyz2 : xyz1, *cols = M > N ? xyz1 : xyz2;
        FEED_CHECK(cudaEventRecord(f->ready, stream));
        FEED_CHECK(cudaStreamWaitEvent(f->copy_stream, f->ready, 0));
        if (!(fuse != nullptr && fuse->workspace_armed)) {
            FEED_CHECK(cudaMemsetAsync(w.packed, 0xff, (n1 + n2) * 8, stream));
            FEED_CHECK(cudaMemsetAsync(w.ctl, 0, 16, stream));
        } else {
            FEED_CHECK(cudaMemsetAsync(w.ctl + 1, 0, 4, stream));   // the chunks OR their verdicts into the selection flag
        }
        FEED_CHECK(cudaEventRecord(f->fork, stream));
        // TWO chunks whatever the caller asked for: a chunk costs ~15 driver calls (copies, events, sort, fork / join of the side
        // stream, scan) and two more streams.  Six chunks were ~90 calls per 0.3-ms step -- as fast as two on a quiet box (0.270 vs
        // 0.260 ms) but 0.69 ms on one of three 2-GPU runs (host-launch bound; 14 streams on 8 hardware queues)
        if (chunks > 2) chunks = 2;
        const int pairs = (B + chunks - 1) / chunks;
        chunks = (B + pairs - 1) / pairs;
        for (int c = 0; c < chunks; ++c) {
            const int b0 = c * pairs, nb = (B - b0 < pairs) ? B - b0 : pairs;
            if (f->cstream[c] == nullptr) FEED_CHECK(cudaStreamCreateWithFlags(&f->cstream[c], cudaStreamNonBlocking));
            FEED_CHECK(cudaMemcpyAsync(xyz1 + (size_t)b0 * N * 3, h_xyz1 + (size_t)b0 * N * 3, (size_t)nb * N * 12,
                                       cudaMemcpyHostToDevice, f->copy_stream));
            FEED_CHECK(cudaMemcpyAsync(xyz2 + (size_t)b0 * M * 3, h_xyz2 + (size_t)b0 * M * 3, (size_t)nb * M * 12,
                                       cudaMemcpyHostToDevice, f->copy_stream));
            FEED_CHECK(cudaEventRecord(f->chunk_ev[c], f->copy_stream));
            FEED_CHECK(cudaStreamWaitEvent(f->cstream[c], f->fork, 0));
            FEED_CHECK(cudaStreamWaitEvent(f->cstream[c], f->chunk_ev[c], 0));
            const int rcs = launch_prune_subbatch(rows, cols, nr_, nc_, w, B, b0, nb, true, f->cstream[c], f->cctl + 4 * c);
            if (rcs != GENPC_OK) return rcs;
            FEED_CHECK(cudaEventRecord(f->done_ev[c], f->cstream[c]));
        }
        for (int c = 0; c < chunks; ++c) FEED_CHECK(cudaStreamWaitEvent(stream, f->done_ev[c], 0));
        const int marker = chunks;
        return chamfer_forward_sym(xyz1, xyz2, dist1, dist2, idx1, idx2, B, N, M, w, stream, nullptr, 0, 1, fuse, &marker);
    }
    const unsigned gen = ++f->gen;
    if (gen % FEED_RING == 0) FEED_CHECK(cudaEventSynchronize(f->copied));  // the ring slot about to be reused has been read
    unsigned *src = f->h_ring + gen % FEED_RING;
    *src = gen;
    // the device buffers may still be read by earlier work on the caller's stream
    FEED_CHECK(cudaEventRecord(f->ready, stream));
    FEED_CHECK(cudaStreamWaitEvent(f->copy_stream, f->ready, 0));
    // ALL copies are queued before the scan is launched: once the kernel is resident and waiting, nothing it needs may
    // depend on further progress of this host thread (a lazily loaded module, a profiler serialising launches or
    // CUDA_LAUNCH_BLOCKING would otherwise turn the wait into a deadlock that only the kernel's timeout breaks)
    for (int c = 0; c < chunks; ++c) {
        const int b0 = c * pairs, nb = (B - b0 < pairs) ? B - b0 : pairs;
        FEED_CHECK(cudaMemcpyAsync(xyz1 + (size_t)b0 * N * 3, h_xyz1 + (size_t)b0 * N * 3, (size_t)nb * N * 12,
                                   cudaMemcpyHostToDevice, f->copy_stream));
        FEED_CHECK(cudaMemcpyAsync(xyz2 + (size_t)b0 * M * 3, h_xyz2 + (size_t)b0 * M * 3, (size_t)nb * M * 12,
                                   cudaMemcpyHostToDevice, f->copy_stream));
        FEED_CHECK(cudaMemcpyAsync(f->gate + c, src, sizeof(unsigned), cudaMemcpyHostToDevice, f->copy_stream));
    }
    const ChamferWs w = chamfer_layout(B, nr_, nc_, 0, workspace);
    if (!(fuse != nullptr && fuse->workspace_armed)) {
        FEED_CHECK(cudaMemsetAsync(w.packed, 0xff, (n1 + n2) * 8, stream));
        FEED_CHECK(cudaMemsetAsync(w.ctl, 0, 16, stream));
    }
    const int rc = chamfer_forward_sym(xyz1, xyz2, dist1, dist2, idx1, idx2, B, N, M, w, stream, f->gate, gen, pairs, fuse);
    if (rc != GENPC_OK) return rc;
    FEED_CHECK(cudaEventRecord(f->copied, f->copy_stream));
    FEED_CHECK(cudaStreamWaitEvent(stream, f->copied, 0));  // later work on the caller's stream sees complete clouds
#undef FEED_CHECK
    return GENPC_OK;
}

// 1 if a gated launch of this feed timed out waiting for its data since the last call of this function (results of that
// launch are invalid; its fused loss, if any, is NaN).  Synchronises `stream`; the error word is cleared once reported.
extern "C" int genpc_host_feed_error(genpc_host_feed_t *f, genpc_stream_t stream_) {
    if (f == nullptr) return GENPC_ERR_SHAPE;
    std::lock_guard<std::mutex> guard(f->lock);
    unsigned v = 0;
    cudaError_t e = cudaMemcpyAsync(&v, f->gate + GATE_ERR_SLOT, sizeof(unsigned), cudaMemcpyDeviceToHost, (cudaStream_t)stream_);
    if (e == cudaSuccess) e = cudaStreamSynchronize((cudaStream_t)stream_);
    if (e == cudaSuccess && v) e = cudaMemsetAsync(f->gate + GATE_ERR_SLOT, 0, sizeof(unsigned), (cudaStream_t)stream_);
    if (e != cudaSuccess) return (int)e;
    return v ? 1 : 0;
}

// Test hook: raise the feed's error word as a timed-out gate would (the 2-second timeout itself cannot be provoked cheaply).
extern "C" int genpc_host_feed_inject_error(genpc_host_feed_t *f, genpc_stream_t stream_) {
    if (f == nullptr) return GENPC_ERR_SHAPE;
    cudaError_t e = cudaMemsetAsync(f->gate + GATE_ERR_SLOT, 1, 1, (cudaStream_t)stream_);
    return e == cudaSuccess ? GENPC_OK : (int)e;
}

// ---- target-sharded Chamfer (million-point clouds over several GPUs) ---------------------------------------
// One direction, one target shard: packed[b][j] = min(packed[b][j], (dist_bits<<32 | idx_base+k)) over the
// targets of this shard.  The caller initialises `packed` to all-ones once (init != 0 does it here), merges the
// shards with an all-reduce-MIN over the 64-bit words (non-negative as int64 because dist >= 0), then unpacks.
extern "C" int genpc_nn_partial_packed(const float *queries, const float *targets_shard, unsigned long long *packed,
                                       int B, int Nq, int Mt_shard, int idx_base, int init, genpc_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (B < 0 || Nq < 0 || Mt_shard < 0 || idx_base < 0) return GENPC_ERR_SHAPE;
    const size_t n1 = (size_t)B * Nq;
    if (n1 == 0) return GENPC_OK;
    if (init) {
        cudaError_t e = cudaMemsetAsync(packed, 0xff, n1 * 8, stream);
        if (e != cudaSuccess) return (int)e;
    }
    if (Mt_shard == 0) return GENPC_OK;
    const int QT = nn_pick_qt(Nq);
    NNParams p;
    fill_dir(p.dir[0], queries, targets_shard, packed, B, Nq, Mt_shard, QT);
    p.dir[0].idx_base = idx_base;
    p.dir[1] = p.dir[0];
    p.dir[1].items = 0;
    if ((long long)p.dir[0].items > 0x7fffffffLL) return GENPC_ERR_RANGE;
    cudaError_t e = QT == 4 ? launch_scan<4>(p, stream) : (QT == 2 ? launch_scan<2>(p, stream) : launch_scan<1>(p, stream));
    if (e != cudaSuccess) return (int)e;
    return GENPC_OK;
}

extern "C" int genpc_nn_unpack(const unsigned long long *packed, float *dist, int *idx, size_t count,
                               genpc_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (count == 0) return GENPC_OK;
    nn_unpack_kernel<<<(unsigned)((count + 255) / 256), 256, 0, stream>>>(const_cast<unsigned long long *>(packed), dist, idx,
                                                                          count, nullptr, nullptr, 0, 0);
    GENPC_CHECK_LAUNCH();
    return GENPC_OK;
}

// ---- row-sharded symmetric Chamfer (multi-GPU, every pair evaluated once across the whole job) ----------------
// Rank r owns rows [row_base, row_base + nr_shard) of cloud 1 (row_base a multiple of 128) and scans them against
// ALL of cloud 2: prow_shard gets the final (dist, idx2) words of its rows, pcol gets (dist, GLOBAL row block)
// partial minima for every point of cloud 2.  pcol is merged across ranks by all-reduce-MIN, then
// genpc_chamfer_sym_fixup resolves the row blocks to exact lowest indices against the FULL cloud 1.
extern "C" int genpc_chamfer_sym_partial(const float *rows_shard, const float *cols, unsigned long long *prow_shard,
                                         unsigned long long *pcol, int B, int nr_shard, int nc, int row_base,
                                         int init_cols, genpc_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (B < 0 || nr_shard < 0 || nc < 0 || row_base < 0 || row_base % 128 != 0) return GENPC_ERR_SHAPE;
    if (B > 1 && row_base != 0) return GENPC_ERR_SHAPE;  // a shard of a batched cloud is not contiguous: B == 1 only
    cudaError_t e;
    if (init_cols && (size_t)B * nc) {
        e = cudaMemsetAsync(pcol, 0xff, (size_t)B * nc * 8, stream);
        if (e != cudaSuccess) return (int)e;
    }
    if ((size_t)B * nr_shard == 0) return GENPC_OK;
    e = cudaMemsetAsync(prow_shard, 0xff, (size_t)B * nr_shard * 8, stream);
    if (e != cudaSuccess) return (int)e;
    if (nc == 0) return GENPC_OK;
    SymParams p = {};
    p.rows = rows_shard, p.cols = cols, p.prow = prow_shard, p.pcol = pcol;
    p.nr = nr_shard, p.nc = nc, p.rblock_base = row_base / 128;
    p.gate = nullptr, p.gate_gen = 0, p.gate_pairs = 1;
    p.select = nullptr;
    const long long items = sym_tiling(B, nr_shard, nc, 4, p.rtiles, p.span, p.cspans);
    if (items > 0x7fffffffLL) return GENPC_ERR_RANGE;
    nn_sym_kernel<4><<<(unsigned)items, SYM_THREADS, 0, stream>>>(p);
    GENPC_CHECK_LAUNCH();
    return GENPC_OK;
}

extern "C" int genpc_chamfer_sym_fixup(const float *rows_full, const float *cols, const unsigned long long *pcol, int B,
                                       int nr_full, int nc, float *dist_cols, int *idx_cols, genpc_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (B < 0 || nr_full < 0 || nc < 0) return GENPC_ERR_SHAPE;
    const size_t ncw = (size_t)B * nc;
    if (ncw == 0) return GENPC_OK;
    // the column half of the forward epilogue alone (no row blocks, nothing fused: pcol is only read)
    EpiFuse f;
    memset(&f, 0, sizeof(f));
    const unsigned fix_blocks = (unsigned)((ncw + EPI_COLS_PER_CTA - 1) / EPI_COLS_PER_CTA);
    nn_sym_epilogue_kernel<false><<<fix_blocks, 256, 0, stream>>>(rows_full, cols, nullptr, const_cast<unsigned long long *>(pcol), B,
                                                                  nr_full, nc, 128, fix_blocks, nullptr, nullptr, dist_cols,
                                                                  idx_cols, f);
    GENPC_CHECK_LAUNCH();
    return GENPC_OK;
}

// ---- fused loss reductions (Completionloss hot calls: utils/loss_util.py:25-43) ----------------------------------
// loss = w1 * mean f(dist1) + w2 * mean f(dist2), f = sqrt (chamfer_l1 / chamfer_partial_l1) or identity (l2 forms).
// One launch, deterministic: fixed-size grid, per-CTA partial sums in double, the last CTA (ticket) adds the partials
// in index order.  Replaces the ~8 tiny torch launches (sqrt, mean, add, div and their backward) per call.
namespace genpc {
constexpr int LOSS_CTAS = 2 * GENPC_NUM_SMS_B200;   // a fixed reduction grid (workspace size depends on it), not a tuning knob

__global__ void __launch_bounds__(256) chamfer_loss_kernel(const float *__restrict__ d1, const float *__restrict__ d2,
                                                           size_t n1, size_t n2, int use_sqrt, float w1, float w2,
                                                           double *partial, unsigned *ticket, float *out) {
    __shared__ double sh[2][8];
    __shared__ int is_last;
    double s1 = 0.0, s2 = 0.0;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n1; i += stride)
        s1 += (double)(use_sqrt ? __fsqrt_rn(__ldg(d1 + i)) : __ldg(d1 + i));
    if (w2 != 0.f)
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += stride)
            s2 += (double)(use_sqrt ? __fsqrt_rn(__ldg(d2 + i)) : __ldg(d2 + i));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s1 += __shfl_xor_sync(0xffffffffu, s1, o), s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) sh[0][warp] = s1, sh[1][warp] = s2;
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
        for (int w = 0; w < 8; ++w) a += sh[0][w], b += sh[1][w];
        partial[2 * blockIdx.x] = a, partial[2 * blockIdx.x + 1] = b;
        __threadfence();
        is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {  // the last CTA adds the per-CTA partials: fixed assignment + fixed tree => deterministic
        __threadfence();
        double a = 0.0, b = 0.0;
        for (unsigned c = threadIdx.x; c < gridDim.x; c += blockDim.x) a += __ldcg(partial + 2 * c), b += __ldcg(partial + 2 * c + 1);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o), b += __shfl_xor_sync(0xffffffffu, b, o);
        __syncthreads();
        if (lane == 0) sh[0][warp] = a, sh[1][warp] = b;
        __syncthreads();
        if (threadIdx.x == 0) {
            a = 0.0, b = 0.0;
            for (int w = 0; w < 8; ++w) a += sh[0][w], b += sh[1][w];
            const double m1 = n1 ? a / (double)n1 : 0.0, m2 = (n2 && w2 != 0.f) ? b / (double)n2 : 0.0;
            out[0] = (float)((double)w1 * m1 + (double)w2 * m2);
            *ticket = 0;
        }
    }
}

}  // namespace genpc

extern "C" size_t genpc_chamfer_loss_workspace_bytes(void) { return (size_t)LOSS_CTAS * 2 * sizeof(double) + 16; }

// workspace must be zero-initialised ONCE by the caller (the ticket word is re-armed by the kernel itself).
extern "C" int genpc_chamfer_loss(const float *dist1, const float *dist2, size_t n1, size_t n2, int use_sqrt, float w1,
                                  float w2, float *out, void *workspace, size_t workspace_bytes, genpc_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (workspace == nullptr || workspace_bytes < genpc_chamfer_loss_workspace_bytes()) return GENPC_ERR_WORKSPACE;
    double *partial = (double *)workspace;
    unsigned *ticket = (unsigned *)(partial + (size_t)LOSS_CTAS * 2);
    chamfer_loss_kernel<<<LOSS_CTAS, 256, 0, stream>>>(dist1, dist2, n1, n2, use_sqrt, w1, w2, partial, ticket, out);
    GENPC_CHECK_LAUNCH();
    return GENPC_OK;
}

// Both loss backward entries; len1 / len2: a ragged batch's lengths, nullptr for an equal-size one.
static int loss_backward(const float *xyz1, const float *xyz2, const int *len1, const int *len2, const float *dist1,
                         const float *dist2, const int *idx1, const int *idx2, const float *upstream, int use_sqrt, float w1,
                         float w2, float *gradxyz1, float *gradxyz2, int B, int N, int M, cudaStream_t stream) {
    if (B < 0 || N < 0 || M < 0) return GENPC_ERR_SHAPE;
    if (N == 0 || M == 0 || B == 0) return GENPC_OK;
    const size_t tot = (size_t)B * N + ((w2 != 0.f) ? (size_t)B * M : 0);
    const bool vec = ((reinterpret_cast<size_t>(gradxyz1) | reinterpret_cast<size_t>(gradxyz2)) & 7) == 0;
    const unsigned grid = (unsigned)((tot + 256 * GRAD_R - 1) / (256 * GRAD_R));
    if (vec)
        chamfer_grad_kernel<true, true><<<grid, 256, 0, stream>>>(xyz1, xyz2, dist1, dist2, idx1, idx2, upstream, use_sqrt, w1, w2,
                                                                 gradxyz1, gradxyz2, B, N, M, len1, len2);
    else
        chamfer_grad_kernel<false, true><<<grid, 256, 0, stream>>>(xyz1, xyz2, dist1, dist2, idx1, idx2, upstream, use_sqrt, w1, w2,
                                                                  gradxyz1, gradxyz2, B, N, M, len1, len2);
    GENPC_CHECK_LAUNCH();
    return GENPC_OK;
}

extern "C" int genpc_chamfer_loss_backward(const float *xyz1, const float *xyz2, const float *dist1, const float *dist2,
                                           const int *idx1, const int *idx2, const float *upstream, int use_sqrt,
                                           float w1, float w2, float *gradxyz1, float *gradxyz2, int B, int N, int M,
                                           genpc_stream_t stream) {
    return loss_backward(xyz1, xyz2, nullptr, nullptr, dist1, dist2, idx1, idx2, upstream, use_sqrt, w1, w2, gradxyz1, gradxyz2, B,
                         N, M, (cudaStream_t)stream);
}

extern "C" int genpc_chamfer_loss_backward_ragged(const float *xyz1, const float *xyz2, const int *len1, const int *len2,
                                                  const float *dist1, const float *dist2, const int *idx1, const int *idx2,
                                                  const float *upstream, int use_sqrt, float w1, float w2, float *gradxyz1,
                                                  float *gradxyz2, int B, int N, int M, genpc_stream_t stream) {
    if (len1 == nullptr || len2 == nullptr) return GENPC_ERR_SHAPE;
    return loss_backward(xyz1, xyz2, len1, len2, dist1, dist2, idx1, idx2, upstream, use_sqrt, w1, w2, gradxyz1, gradxyz2, B, N,
                         M, (cudaStream_t)stream);
}
