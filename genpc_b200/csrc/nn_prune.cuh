// nn_prune.cuh -- exact nearest neighbours with spatial pruning (r02).  The default Chamfer scan for batches (device-resident or
// host-fed) of >= 2^30 distance evaluations (BASELINE C2) and inside the registration loop from ~20 scans up; the sort kernel also serves the
// EMD auction's pruned Bid.  GENPC_CHAMFER_PRUNE / GENPC_REGISTER_PRUNE = 0 / 1 forbid / force it.
//
// The symmetric scan (nn_sym.cuh) evaluates every (row, column) distance of a cloud pair: at its issue limit that is
// 7.9e12 pairs/s and nothing in its instruction stream is left to remove.  What is left is not to evaluate most pairs:
//   1. nn_bin_sort_kernel<CS> orders every cloud along a Hilbert curve (counting sort over 8^m grid cells in shared memory;
//      one CTA per cloud, or a thread-block cluster of CS CTAs that read each other's histograms through distributed shared
//      memory when one CTA per cloud would leave most SMs idle) into (x, y, z, original index) records and stores the
//      bounding box of every PR_BLOCK consecutive ones, and of every 8 (the walk's chunks);
//   2. nn_prune_kernel: one warp owns PR_GROUP consecutive sorted queries (one per lane -- neighbours in space).  It
//      computes the squared distance between the group's box and every target block's box, visits the blocks nearest
//      first (REDUX picks them) and stops at the first block farther than the group's worst running minimum: no target
//      in it, or in any later block, can improve (or tie) any lane.  A block is fetched only when some lane's own point is
//      within its box, with one coalesced read into the warp's shared-memory slice (SoA), and walked there chunk by chunk
//      with the packed FP32 distance of the exhaustive kernels (the same bits), skipping the chunks whose box no lane is
//      within (pr_visit_block).  nn_prune_coop_kernel is the form for a direction with few query groups and many target blocks: a CTA
//      per group, the blocks partitioned over its eight warps, running minima shared through shared memory.
// Exactness: the minimum of a set does not depend on the visiting order; the reported index is the LOWEST original index
// among the targets at the minimum, as in the exhaustive kernels (the winner's 8-target chunk is re-evaluated; a lane
// that saw the same minimum in two chunks takes a second pass over the surviving blocks).  The box distance is scaled
// down by 1e-5, far more than the rounding of the reference's arithmetic, and compared with <= so that ties are kept.
// The sort kernel doubles as the range check (NaN / Inf / |x| > 1e15 -> the exhaustive kernel runs instead, selected on
// the device through a flag in the control words that the exhaustive kernel and the epilogue read).
#pragma once
#include <cooperative_groups.h>

#include <type_traits>

#include "common.cuh"
#include "nn_core.cuh"   // Similarity / apply_similarity (registration: the moving cloud is sorted in its current pose)

#ifndef GENPC_PR_UNROLL
#define GENPC_PR_UNROLL 4   // 8-target chunks per unrolled step of a block walk (sweep 1/2/4/8: profiles/r02w_unroll_sweep.txt)
#endif

namespace genpc {

constexpr int PR_UNROLL = GENPC_PR_UNROLL;
constexpr int PR_BLOCK = 64;
constexpr int PR_GROUP = 32;
constexpr int PR_MAX_N = 32768;       // 512 blocks: the block id fits the 9 low bits of the selection key
constexpr int PR_SORT_THREADS = 1024;
constexpr int PR_MAX_CELLS = 4096;
constexpr int PR_THREADS = 256;

__host__ __device__ inline int pr_nblk(int n) { return (n + PR_BLOCK - 1) / PR_BLOCK; }
__host__ __device__ inline int pr_npad(int n) { return pr_nblk(n) * PR_BLOCK; }

// Calls f(std::integral_constant<int, R>()) with the rows R = 1 / 2 / 4 / 8 / 16 of 32 box distances that a lane of the pruned
// kernels keeps in registers for `n` target blocks (or superblocks): the smallest R with R * 32 >= n
template <typename F>
static void pr_rows(int n, F &&f) {
    if (n <= 32) f(std::integral_constant<int, 1>());
    else if (n <= 64) f(std::integral_constant<int, 2>());
    else if (n <= 128) f(std::integral_constant<int, 4>());
    else if (n <= 256) f(std::integral_constant<int, 8>());
    else f(std::integral_constant<int, 16>());
}

// 3 * BITS-bit Hilbert index of a grid cell (Skilling, "Programming the Hilbert curve", 2004: axes -> transpose -> interleave).
// Consecutive indices are always neighbouring cells, so ANY run of consecutive sorted points is spatially connected; a
// Morton (Z-order) run that crosses a high-level cell boundary joins two far-apart regions in one bounding box, and every
// query group inside that box has to open it (the first r02 form: 59 instead of ~10 block visits per group on the LiDAR scene).
template <int BITS>
__device__ __forceinline__ unsigned hilbert_key(unsigned x, unsigned y, unsigned z) {
    unsigned X[3] = {x, y, z};
    constexpr unsigned M = 1u << (BITS - 1);
#pragma unroll
    for (unsigned Q = M; Q > 1; Q >>= 1) {
        const unsigned P = Q - 1;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            if (X[i] & Q) {
                X[0] ^= P;
            } else {
                const unsigned t = (X[0] ^ X[i]) & P;
                X[0] ^= t, X[i] ^= t;
            }
        }
    }
    X[1] ^= X[0], X[2] ^= X[1];
    unsigned t = 0;
#pragma unroll
    for (unsigned Q = M; Q > 1; Q >>= 1)
        if (X[2] & Q) t ^= Q - 1;
    X[0] ^= t, X[1] ^= t, X[2] ^= t;
    unsigned key = 0;
#pragma unroll
    for (int j = BITS - 1; j >= 0; --j)
#pragma unroll
        for (int i = 0; i < 3; ++i) key = (key << 1) | ((X[i] >> j) & 1u);
    return key;
}

struct PruneSortParams {
    const float *xyz[2];   // [B][n][3]
    float4 *sorted[2];     // [B][npad]   (x, y, z, original index); NaN records pad the last block
    float4 *boxes[2];      // [B][2][nblk] lower corners, then upper corners
    float4 *cboxes[2];     // optional [B][2][npad / 8]: the same for every 8 consecutive records (the scan's chunks; nullptr: none)
    int n[2];
    int B;
    float limit;
    int *ctl;              // [1] selection flag (0: pruned kernels run), [2] accumulator, [3] ticket of the range check
    int hilbert;           // cell order: Hilbert curve (1) or Z-order (0)
    float *bbx;            // optional [2][B][8]: every cloud's bounding box, for the overlap test below (nullptr: none)
    int accumulate;        // 1: OR the verdict into ctl[1] (a later chunk of the same batch), 0: overwrite it
    int *flag;             // optional: atomicOr the verdict here instead (chunks sorted concurrently on several streams; ctl then
                           // only provides the chunk's own accumulator / ticket words)
    // registration: only one side is sorted per launch (side0 = its index, grid = B), its points taken from cloud b / src_div
    // and moved by the similarity sim[b] while they are read (the same rounding as the exhaustive scan's staging)
    int side0, single_side;
    int mixed;             // cluster launches only: the larger side's clouds take a whole cluster each, the other side's one CTA each
    int src_div[2];
    const Similarity *sim[2];
};

// <<<ctas, 256>>>: all-ones into the packed words when the selection flag asks for the exhaustive kernels AFTER pruned launches
// have already stored exact (dist, index) words (chunked host-fed batches: a later chunk may be the one out of range)
static __global__ void prune_rearm_kernel(unsigned long long *words, size_t n, const int *select) {
    if (*select == 0) return;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) words[i] = ~0ull;
}

// grid = 2 * B * CS CTAs: cloud = blockIdx.x / CS = side * B + b (or the mixed layout below).  CS > 1 (launched as thread-block
// clusters of CS CTAs): the CTAs of a cluster share one cloud -- every CTA takes each CS-th slab of 1024 points, keeps its own
// histogram, and reads its siblings'
// bounding boxes and histograms through distributed shared memory (a point's slot = cells before it + the same cell's counts in
// the lower-ranked CTAs + the CTA's own atomic counter); the block boxes are split between the CTAs after the last cluster
// barrier.  One CTA per 16384-point cloud was 55 us of C2's 170 us forward with 84 of the 148 SMs idle.
template <int CS>
static __global__ void __launch_bounds__(PR_SORT_THREADS) nn_bin_sort_kernel(const PruneSortParams p) {
    cudaTriggerProgrammaticLaunchCompletion();   // the pruned scan behind it (launch_pdl) may take the SMs the sort leaves free
    __shared__ __align__(16) int hist[PR_MAX_CELLS];
    __shared__ __align__(16) int slot[CS > 1 ? PR_MAX_CELLS : 4];   // CS > 1: next free slot per cell (hist stays readable for the siblings)
    __shared__ float sred[6][PR_SORT_THREADS / 32];
    __shared__ float cbox[8];
    __shared__ int swarp[PR_SORT_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // cr = rank of this CTA among the `ceff` CTAs that share its cloud, r0 = cluster rank of the first of them
    int cr = 0, r0 = 0, ceff = 1, cloud = (int)blockIdx.x;
    bool idle = false;
    if constexpr (CS > 1) {
        const int rank = (int)cooperative_groups::this_cluster().block_rank();
        if (p.mixed) {
            // clusters [0, B): one cloud of the LARGER side each; the CTAs behind them: one cloud of the other side each, on their
            // own (they only keep the cluster barriers company); CTAs that round the grid up to whole clusters idle
            const int big = p.n[1] > p.n[0] ? 1 : 0;
            if ((int)blockIdx.x < p.B * CS) {
                cloud = big * p.B + (int)blockIdx.x / CS, cr = rank, ceff = CS;
            } else {
                const int j = (int)blockIdx.x - p.B * CS;
                idle = j >= p.B;
                cloud = (1 - big) * p.B + (idle ? 0 : j), r0 = rank;
            }
        } else {
            cloud = (int)blockIdx.x / CS, cr = rank, ceff = CS;
        }
    }
    const int side = p.single_side ? p.side0 : cloud / p.B, b = cloud % p.B;
    const int STRIDE = ceff * PR_SORT_THREADS;
    const int n = idle ? 0 : p.n[side], nblk = pr_nblk(n), npad = nblk * PR_BLOCK;
    const float *src = p.xyz[side] + (size_t)(p.src_div[side] > 1 ? b / p.src_div[side] : b) * n * 3;
    __shared__ Similarity sT;
    const bool moved = p.sim[side] != nullptr;
    if (moved && tid == 0) sT = p.sim[side][b];
    if (moved) __syncthreads();
    auto load_point = [&](int k, float &x, float &y, float &z) {
        x = __ldg(src + k * 3), y = __ldg(src + k * 3 + 1), z = __ldg(src + k * 3 + 2);
        if (moved) apply_similarity(sT, x, y, z);
    };
    float4 *dst = p.sorted[side] + (size_t)b * npad;
    float4 *bx = p.boxes[side] + (size_t)b * 2 * nblk;
    const float inf = __int_as_float(0x7f800000);
    // ---- bounding box + range check ----
    float lo[3] = {inf, inf, inf}, hi[3] = {-inf, -inf, -inf};
    bool bad = false;
    for (int k = cr * PR_SORT_THREADS + tid; k < n; k += STRIDE) {
        float v[3];
        load_point(k, v[0], v[1], v[2]);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            bad |= !(fabsf(v[c]) <= p.limit);
            lo[c] = fminf(lo[c], v[c]), hi[c] = fmaxf(hi[c], v[c]);
        }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[c] = fminf(lo[c], __shfl_xor_sync(0xffffffffu, lo[c], o));
            hi[c] = fmaxf(hi[c], __shfl_xor_sync(0xffffffffu, hi[c], o));
        }
        if (lane == 0) sred[c][warp] = lo[c], sred[3 + c][warp] = hi[c];
    }
#ifndef GENPC_SORT_BITS4_FROM
#define GENPC_SORT_BITS4_FROM 2048   // 16^3 cells from 2048 points up (5 % fewer block visits on C2 than 8^3 cells for the 2048-point clouds)
#endif
    int mbits = n >= GENPC_SORT_BITS4_FROM ? 4 : (n >= 1024 ? 3 : (n >= 128 ? 2 : 1));
    const int ncell = 1 << (3 * mbits);
    for (int k = tid; k < ncell; k += PR_SORT_THREADS) hist[k] = 0;
    const int anybad = __syncthreads_or(bad ? 1 : 0);
    float scale[3];
    if constexpr (CS > 1) {   // the cloud's box = the union of the CTAs' boxes
        if (tid < 6) {
            float r = tid < 3 ? inf : -inf;
            for (int w = 0; w < PR_SORT_THREADS / 32; ++w) r = tid < 3 ? fminf(r, sred[tid][w]) : fmaxf(r, sred[tid][w]);
            cbox[tid] = r;
        }
        cooperative_groups::cluster_group cluster = cooperative_groups::this_cluster();
        cluster.sync();
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float l = inf, h = -inf;
            for (int r = r0; r < r0 + ceff; ++r) {
                const float *o = cluster.map_shared_rank(cbox, r);
                l = fminf(l, o[c]), h = fmaxf(h, o[3 + c]);
            }
            lo[c] = l, hi[c] = h;
        }
    } else {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float l = inf, h = -inf;
            for (int w = 0; w < PR_SORT_THREADS / 32; ++w) l = fminf(l, sred[c][w]), h = fmaxf(h, sred[3 + c][w]);
            lo[c] = l, hi[c] = h;
        }
    }
    if (tid == 0 && cr == 0 && !idle && p.bbx != nullptr) {   // read by the last CTA of the grid, behind its ticket (below)
        float *o = p.bbx + ((size_t)side * p.B + b) * 8;
        for (int c = 0; c < 3; ++c) o[c] = lo[c], o[3 + c] = hi[c];
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float ext = hi[c] - lo[c];
        scale[c] = (ext > 0.f && ext < inf) ? (float)(1 << mbits) / ext : 0.f;
    }
    const int cmax = (1 << mbits) - 1;
    const bool hilbert = p.hilbert != 0;
    auto cell_of = [&](int k, float &x, float &y, float &z) {
        load_point(k, x, y, z);
        const float v[3] = {x, y, z};
        unsigned code = 0;
        unsigned cc[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float f = (v[c] - lo[c]) * scale[c];
            cc[c] = f >= 0.f ? (unsigned)min((int)fminf(f, 2e9f), cmax) : 0u;
        }
        if (hilbert) {   // connected runs: tighter block boxes than the Z-order below
            code = mbits == 4 ? hilbert_key<4>(cc[0], cc[1], cc[2]) : mbits == 3 ? hilbert_key<3>(cc[0], cc[1], cc[2])
                 : mbits == 2 ? hilbert_key<2>(cc[0], cc[1], cc[2]) : hilbert_key<1>(cc[0], cc[1], cc[2]);
            return (int)code;
        }
        for (int bit = 0; bit < mbits; ++bit)
#pragma unroll
            for (int c = 0; c < 3; ++c) code |= (unsigned)((cc[c] >> bit) & 1) << (3 * bit + c);
        return (int)code;
    };
    // ---- histogram; clouds of up to 16384 points keep each point's cell in registers for the scatter pass (the Hilbert key is
    // a third of this kernel's instructions when it is computed in both passes) ----
    constexpr int KEEP = CS == 1 ? 16 : (PR_MAX_N + CS * PR_SORT_THREADS - 1) / (CS * PR_SORT_THREADS);   // CS > 1: every size up to PR_MAX_N
    const bool keep = n <= KEEP * STRIDE;
    unsigned short cells[KEEP];
    if (keep) {
#pragma unroll
        for (int i = 0; i < KEEP; ++i) {
            const int k = cr * PR_SORT_THREADS + tid + i * STRIDE;
            cells[i] = 0;
            if (k < n) {
                float x, y, z;
                cells[i] = (unsigned short)cell_of(k, x, y, z);
                atomicAdd(&hist[cells[i]], 1);
            }
        }
    } else {
        for (int k = cr * PR_SORT_THREADS + tid; k < n; k += STRIDE) {
            float x, y, z;
            atomicAdd(&hist[cell_of(k, x, y, z)], 1);
        }
    }
    if constexpr (CS > 1) cooperative_groups::this_cluster().sync();   // every sibling's histogram is complete
    else __syncthreads();
    // ---- exclusive scan of the histogram (4 entries per thread; CS > 1: of the sum of the CS histograms) ----
    int *next = CS > 1 ? slot : hist;
    {
        constexpr int per = PR_MAX_CELLS / PR_SORT_THREADS;
        static_assert(per == 4, "one int4 of cells per thread");
        int v[per], below[per], s = 0;
#pragma unroll
        for (int i = 0; i < per; ++i) v[i] = below[i] = 0;
        if (tid * per < ncell) {   // ncell is 8, 64, 512 or 4096: a thread's four cells are all inside or all outside
            if constexpr (CS > 1) {
                cooperative_groups::cluster_group cluster = cooperative_groups::this_cluster();
                for (int r = r0; r < r0 + ceff; ++r) {
                    const int4 t = *reinterpret_cast<const int4 *>(cluster.map_shared_rank(hist, r) + tid * per);
                    const int tv[per] = {t.x, t.y, t.z, t.w};
#pragma unroll
                    for (int i = 0; i < per; ++i) {
                        v[i] += tv[i];
                        if (r < r0 + cr) below[i] += tv[i];
                    }
                }
            } else {
                const int4 t = *reinterpret_cast<const int4 *>(hist + tid * per);
                v[0] = t.x, v[1] = t.y, v[2] = t.z, v[3] = t.w;
            }
        }
#pragma unroll
        for (int i = 0; i < per; ++i) s += v[i];
        int incl = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) swarp[warp] = incl;
        __syncthreads();
        int base = 0;
        for (int w = 0; w < warp; ++w) base += swarp[w];
        int run = base + incl - s;
#pragma unroll
        for (int i = 0; i < per; ++i) {
            const int e = tid * per + i;
            if (e < ncell) next[e] = run + below[i];
            run += v[i];
        }
    }
    __syncthreads();
    // ---- scatter (the order inside a cell is whatever the atomics give: it only shapes the blocks, never a result) ----
    if (keep) {
#pragma unroll
        for (int i = 0; i < KEEP; ++i) {
            const int k = cr * PR_SORT_THREADS + tid + i * STRIDE;
            if (k < n) {
                float x, y, z;
                load_point(k, x, y, z);
                const int pos = atomicAdd(&next[cells[i]], 1);
                dst[pos] = make_float4(x, y, z, __int_as_float(k));
            }
        }
    } else {
        for (int k = cr * PR_SORT_THREADS + tid; k < n; k += STRIDE) {
            float x, y, z;
            const int cell = cell_of(k, x, y, z);
            const int pos = atomicAdd(&next[cell], 1);
            dst[pos] = make_float4(x, y, z, __int_as_float(k));
        }
    }
    const float qnan = __int_as_float(0x7fc00000);
    if (cr == 0)
        for (int k = n + tid; k < npad; k += PR_SORT_THREADS) dst[k] = make_float4(qnan, qnan, qnan, __int_as_float(0));
    if constexpr (CS > 1) {
        // the siblings' records are read below: fence + cluster barrier, and the loads bypass L1 (__ldcg).  The barrier also is
        // the last point at which a sibling reads this CTA's shared memory: nobody exits before it
        __threadfence();
        cooperative_groups::this_cluster().sync();
    } else {
        __syncthreads();   // the CTA's own global writes are visible to it after the barrier
    }
    // ---- block boxes, and the boxes of the 8-record chunks (the 8-lane stage of the same reduction) ----
    static_assert(PR_BLOCK == 64, "a block is two 32-record rows of the warp");
    float4 *cbx = p.cboxes[side] != nullptr ? p.cboxes[side] + (size_t)b * 2 * (npad / 8) : nullptr;
    for (int blk = cr * (PR_SORT_THREADS / 32) + warp; blk < nblk; blk += ceff * (PR_SORT_THREADS / 32)) {
        float l[PR_BLOCK / 32][3], h[PR_BLOCK / 32][3];
#pragma unroll
        for (int e = 0; e < PR_BLOCK / 32; ++e) {
            const float4 t = CS > 1 ? __ldcg(dst + blk * PR_BLOCK + e * 32 + lane) : dst[blk * PR_BLOCK + e * 32 + lane];
            // NaN padding is ignored: an all-padding chunk keeps (+inf, -inf), a box no point is near
            l[e][0] = fminf(inf, t.x), h[e][0] = fmaxf(-inf, t.x);
            l[e][1] = fminf(inf, t.y), h[e][1] = fmaxf(-inf, t.y);
            l[e][2] = fminf(inf, t.z), h[e][2] = fmaxf(-inf, t.z);
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int o = 4; o > 0; o >>= 1) {
                    l[e][c] = fminf(l[e][c], __shfl_xor_sync(0xffffffffu, l[e][c], o));
                    h[e][c] = fmaxf(h[e][c], __shfl_xor_sync(0xffffffffu, h[e][c], o));
                }
            if (cbx != nullptr && (lane & 7) == 0) {   // records e * 32 + lane .. + 7 of the block: its chunk e * 4 + lane / 8
                const int k = blk * (PR_BLOCK / 8) + e * 4 + (lane >> 3);
                cbx[k] = make_float4(l[e][0], l[e][1], l[e][2], 0.f), cbx[npad / 8 + k] = make_float4(h[e][0], h[e][1], h[e][2], 0.f);
            }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            l[0][c] = fminf(l[0][c], l[1][c]), h[0][c] = fmaxf(h[0][c], h[1][c]);
#pragma unroll
            for (int o = 16; o > 4; o >>= 1) {
                l[0][c] = fminf(l[0][c], __shfl_xor_sync(0xffffffffu, l[0][c], o));
                h[0][c] = fmaxf(h[0][c], __shfl_xor_sync(0xffffffffu, h[0][c], o));
            }
        }
        if (lane == 0)
            bx[blk] = make_float4(l[0][0], l[0][1], l[0][2], 0.f), bx[nblk + blk] = make_float4(h[0][0], h[0][1], h[0][2], 0.f);
    }
    // ---- selection flag: the last CTA publishes "any cloud out of range, or a pair of clouds that does not overlap" (pruning
    // needs neighbours to be near: when the two boxes of a pair are further apart than a quarter of the smaller one's diagonal,
    // or one box is less than a quarter of the other across, every query group would open every block, 2.8x the cost of the
    // exhaustive scan) ----
    if (tid == 0) {
        if (anybad) atomicOr(p.ctl + 2, 1);
        __threadfence();
        if (atomicAdd(p.ctl + 3, 1) == (int)gridDim.x - 1) {
            __threadfence();
            int apart = 0;
            if (p.bbx != nullptr && !p.single_side) {
                for (int i = 0; i < p.B; ++i) {
                    const volatile float *u = p.bbx + (size_t)i * 8, *v = p.bbx + ((size_t)p.B + i) * 8;
                    float gap2 = 0.f, du = 0.f, dv = 0.f;
                    for (int c = 0; c < 3; ++c) {
                        const float g = fmaxf(fmaxf(u[c] - v[3 + c], v[c] - u[3 + c]), 0.f);
                        gap2 += g * g, du += (u[3 + c] - u[c]) * (u[3 + c] - u[c]), dv += (v[3 + c] - v[c]) * (v[3 + c] - v[c]);
                    }
                    if (gap2 > 0.0625f * fminf(du, dv)) apart = 1;
                    // ... and a cloud collapsed to a blob next to a spread-out one (an untrained generator's output against its
                    // target): every group of the large cloud finds all blocks of the blob equally near and opens them all
                    if (fminf(du, dv) < 0.0625f * fmaxf(du, dv)) apart = 1;
                }
            }
            const int verdict = atomicExch(p.ctl + 2, 0) | apart;
            if (p.flag != nullptr) {
                if (verdict) atomicOr(p.flag, 1);
            } else {
                p.ctl[1] = p.accumulate ? (p.ctl[1] | verdict) : verdict;
            }
            p.ctl[3] = 0;
        }
    }
}

// The sort's outputs (sorted records, block boxes, chunk boxes) for clouds[i] clouds of n[i] points on side i of a pruned scan
static inline PruneSortParams pr_take_sorted(WsCursor &c, const int clouds[2], const int n[2]) {
    PruneSortParams sp = {};
    for (int i = 0; i < 2; ++i) sp.n[i] = n[i], sp.sorted[i] = c.take<float4>((size_t)clouds[i] * pr_npad(n[i]));
    for (int i = 0; i < 2; ++i) sp.boxes[i] = c.take<float4>((size_t)clouds[i] * 2 * pr_nblk(n[i]));
    for (int i = 0; i < 2; ++i) sp.cboxes[i] = c.take<float4>((size_t)clouds[i] * 2 * (pr_npad(n[i]) / 8));
    return sp;
}

// `ctas` CTAs (rounded up to whole clusters) as thread-block clusters of CS
template <int CS>
static void launch_bin_sort_cs(PruneSortParams sp, int ctas, cudaStream_t stream) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)((ctas + CS - 1) / CS * CS));
    cfg.blockDim = dim3(PR_SORT_THREADS);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS, attr[0].val.clusterDim.y = 1, attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr, cfg.numAttrs = 1;
    if (cudaLaunchKernelEx(&cfg, nn_bin_sort_kernel<CS>, sp) != cudaSuccess) {
        // a part whose GPCs cannot co-schedule CS 1024-thread CTAs (MIG slices, harvested parts): one CTA per cloud
        (void)cudaGetLastError();
        sp.mixed = 0;
        nn_bin_sort_kernel<1><<<(sp.single_side ? 1 : 2) * sp.B, PR_SORT_THREADS, 0, stream>>>(sp);
    }
}


struct PruneParams {
    const float4 *q, *t;      // sorted queries [B][npad_q], sorted targets [B][npad_t]
    const float4 *tbox;       // [B][2][nblk_t]
    const float4 *tcbox;      // [B][2][npad_t / 8]: boxes of the targets' 8-record chunks
    unsigned long long *out;  // [B][nq] packed (dist, original target index), addressed by the query's original index
    int nq, nt, B;
    const int *select;        // run only when *select == 0
    unsigned *stats;          // optional [4]: blocks fetched and walked, tie passes, groups, 8-target chunks evaluated
    int qdiv, tdiv;           // batch entry b reads queries / targets of cloud b / qdiv, b / tdiv (0 or 1: its own; registration: the
                              // starts of one scan share the fixed cloud's sorted copy)
};

__device__ __forceinline__ int pr_f2ord(float f) {
    const int i = __float_as_int(f);
    return i ^ ((i >> 31) & 0x7fffffff);
}
__device__ __forceinline__ float pr_ord2f(int i) { return __int_as_float(i ^ ((i >> 31) & 0x7fffffff)); }

// Squared distance between the box [l, h] (a query group's box, or one query: l = h) and a target box [lo, hi], scaled down
// (see the header).  Every step rounds monotonically, so it never exceeds the rounded distance (sqdist_ref) of any point of the
// first box to any point of the second.
__device__ __forceinline__ float pr_box_d2(float lx, float ly, float lz, float hx, float hy, float hz, float4 lo, float4 hi) {
    const float dx = fmaxf(fmaxf(lo.x - hx, lx - hi.x), 0.f);
    const float dy = fmaxf(fmaxf(lo.y - hy, ly - hi.y), 0.f);
    const float dz = fmaxf(fmaxf(lo.z - hz, lz - hi.z), 0.f);
    return __fmul_rn(__fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy))), 0.99999f);
}

// One visit of target block `blk` by a warp's 32 queries (one per lane; nx/ny/nz = the negated query in both halves; CBL = the
// lane's entry of chunk box 0 for lanes 0-15).  A lane's bound is min(best, cap): its running minimum, or less when another
// warp has already found a nearer target for the same query (cap; +inf for a warp on its own).
//   1. each lane's point-to-block-box distance against its bound: when no lane is within it, nothing is fetched (-> false);
//   2. the block's 64 records (SoA) and its eight chunk boxes into the warp's staging slice: one coalesced 1 KB + 256 B read;
//   3. each 8-target chunk is evaluated only when some lane's point-to-chunk-box distance is within that lane's CURRENT bound.
// Exactness: a chunk (or block) is skipped only when, for every lane, the box distance is strictly greater than the bound.  The
// box distance is never above the distance the lane would compute to any target inside (pr_box_d2), and the bound is never
// below the lane's current or final minimum, so a skipped chunk could neither lower `best` nor equal it: best, bchunk and tie are
// those of walking every chunk, and a chunk holding a lane's final minimum is always evaluated.  Lanes without a query (padding)
// ask for nothing.
template <int UNR>
__device__ __forceinline__ bool pr_visit_block(float (*st)[PR_BLOCK], float4 *sbox, const float4 *T, const float4 *BL, const float4 *BH,
                                               const float4 *CBL, int blk, float2 nx, float2 ny, float2 nz, bool valid,
                                               float cap, float &best, int &bchunk, bool &tie, unsigned &chunks) {
    const int lane = threadIdx.x & 31;
    const float qx = -nx.x, qy = -ny.x, qz = -nz.x;
    const float inf = __int_as_float(0x7f800000);
    // (`&`, not `&&`: the test is computed by every lane, no branch around it)
    if (!__any_sync(0xffffffffu, valid & (pr_box_d2(qx, qy, qz, qx, qy, qz, __ldg(BL + blk), __ldg(BH + blk)) <= fminf(best, cap))))
        return false;
    {   // one coalesced read of the records, lanes 0-15 the chunk boxes (lower corners, then upper), walked in shared memory
        const float4 *tg = T + blk * PR_BLOCK;
        const float4 u0 = __ldg(tg + lane), u1 = __ldg(tg + 32 + lane);
        const float4 cb = lane < 16 ? __ldg(CBL + blk * (PR_BLOCK / 8)) : make_float4(0.f, 0.f, 0.f, 0.f);
        __syncwarp();
        st[0][lane] = u0.x, st[1][lane] = u0.y, st[2][lane] = u0.z;
        st[0][32 + lane] = u1.x, st[1][32 + lane] = u1.y, st[2][32 + lane] = u1.z;
        if (lane < 16) sbox[lane] = cb;
        __syncwarp();
    }
    // SoA: one LDS.128 per coordinate brings four targets as two register pairs the packed FP32 instructions take as they
    // are (the AoS form spent 6 of its 15 instructions per target pair moving registers into pairs)
    const float4 *sx4 = reinterpret_cast<const float4 *>(st[0]), *sy4 = reinterpret_cast<const float4 *>(st[1]),
                 *sz4 = reinterpret_cast<const float4 *>(st[2]);
#pragma unroll UNR
    for (int c = 0; c < PR_BLOCK / 8; ++c) {
        if (!__any_sync(0xffffffffu, valid & (pr_box_d2(qx, qy, qz, qx, qy, qz, sbox[c], sbox[8 + c]) <= fminf(best, cap)))) continue;
        ++chunks;
        float cm = inf;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const float4 X = sx4[c * 2 + i], Y = sy4[c * 2 + i], Z = sz4[c * 2 + i];
            const float2 a2 = sqdist_ref_x2(nx, ny, nz, make_float2(X.x, X.y), make_float2(Y.x, Y.y), make_float2(Z.x, Z.y));
            const float2 b2 = sqdist_ref_x2(nx, ny, nz, make_float2(X.z, X.w), make_float2(Y.z, Y.w), make_float2(Z.z, Z.w));
            cm = fmin3(cm, a2.x, a2.y);
            cm = fmin3(cm, b2.x, b2.y);
        }
        if (cm < best) {
            best = cm, bchunk = blk * (PR_BLOCK / 8) + c, tie = false;
        } else if (cm == best && cm < inf) {
            tie = true;
        }
    }
    return true;
}

// Both directions of a cloud pair in ONE launch: the first ctas0 CTAs take direction d[0] (put the direction with the longer
// per-group chains there: it is scheduled first), the rest d[1].
struct PrunePair {
    PruneParams d[2];
    int ctas0;
};

// grid = sum over the two directions of B * ceil(groups / 8) CTAs of 8 warps; BOXR * 32 >= nblk of either target cloud
template <int BOXR>
__global__ void __launch_bounds__(PR_THREADS) nn_prune_kernel(const PrunePair pp) {
    __shared__ __align__(16) float stage[PR_THREADS / 32][3][PR_BLOCK];   // the block being walked, SoA: x[64] y[64] z[64]
    __shared__ float4 sbox[PR_THREADS / 32][16];                           // ... and its chunk boxes: lower corners, upper corners
    const int dir = (int)blockIdx.x >= pp.ctas0 ? 1 : 0;
    const PruneParams &p = pp.d[dir];
    cudaGridDependencySynchronize();   // launched behind the sort (pr_launch): its records, boxes and selection flag are complete
    cudaTriggerProgrammaticLaunchCompletion();
    if (p.select != nullptr && *p.select != 0) return;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int groups = (p.nq + PR_GROUP - 1) / PR_GROUP;
    const int ctas_per_cloud = (groups + PR_THREADS / 32 - 1) / (PR_THREADS / 32);
    const int bx = (int)blockIdx.x - dir * pp.ctas0;
    const int b = bx / ctas_per_cloud;
    const int g = (bx % ctas_per_cloud) * (PR_THREADS / 32) + wid;
    if (g >= groups) return;
    const int nblk = pr_nblk(p.nt);
    const int bt = p.tdiv > 1 ? b / p.tdiv : b, bq = p.qdiv > 1 ? b / p.qdiv : b;
    const float4 *T = p.t + (size_t)bt * pr_npad(p.nt);
    const float4 *BL = p.tbox + (size_t)bt * 2 * nblk, *BH = BL + nblk;
    const int nchunk = pr_npad(p.nt) / 8;   // lanes 0-7 / 8-15 stage the lower / upper corners of a block's eight chunk boxes
    const float4 *CBL = p.tcbox + (size_t)bt * 2 * nchunk + (lane >> 3) * nchunk + (lane & 7);
    const float inf = __int_as_float(0x7f800000);
    const int qi = g * PR_GROUP + lane;
    const bool valid = qi < p.nq;
    const float4 q = p.q[(size_t)bq * pr_npad(p.nq) + qi];   // the padding records are NaN: they never win, nothing is stored
    // ---- the group's box ----
    float glo[3], ghi[3];
    {
        const float v[3] = {q.x, q.y, q.z};
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            // NaN (padding) must not take part: +inf / -inf are neutral
            const float a = valid ? v[c] : inf, z = valid ? v[c] : -inf;
            glo[c] = pr_ord2f(__reduce_min_sync(0xffffffffu, pr_f2ord(a)));
            ghi[c] = pr_ord2f(__reduce_max_sync(0xffffffffu, pr_f2ord(z)));
        }
    }
    // ---- squared box-to-box distances, scaled down (see the header) ----
    float bd[BOXR];
#pragma unroll
    for (int r = 0; r < BOXR; ++r) {
        const int blk = r * 32 + lane;
        bd[r] = inf;
        if (blk < nblk) bd[r] = pr_box_d2(glo[0], glo[1], glo[2], ghi[0], ghi[1], ghi[2], __ldg(BL + blk), __ldg(BH + blk));
    }
    const float2 nx = make_float2(-q.x, -q.x), ny = make_float2(-q.y, -q.y), nz = make_float2(-q.z, -q.z);
    float best = inf;
    int bchunk = 0;
    bool tie = false;
    float thr = inf;   // the largest running minimum of the group's lanes
    unsigned scanned = 0, chunks = 0;
    for (;;) {
        // nearest remaining block: (distance bits without the low 9, block id); the truncation errs on the near side
        unsigned key = 0xffffffffu;
#pragma unroll
        for (int r = 0; r < BOXR; ++r) key = min(key, (__float_as_uint(bd[r]) & 0xfffffe00u) | (unsigned)(r * 32 + lane));
        key = __reduce_min_sync(0xffffffffu, key);
        if (key >= 0x7f800000u || !(__uint_as_float(key & 0xfffffe00u) <= thr)) break;
        const int blk = (int)(key & 0x1ffu);
#pragma unroll
        for (int r = 0; r < BOXR; ++r)
            if (r * 32 + lane == blk) bd[r] = inf;
        // 256 target blocks and more (C3: 16384^2 inside the registration loop) keep the 2x form: 4x cost C3 9 % on the same box
        // (26 100 vs 28 600 scan-iters/s) while the 32- and 128-block instantiations gained 1-4 % (profiles/r02w_unroll_sweep.txt)
        constexpr int UNR = BOXR >= 8 ? 2 : PR_UNROLL;
        if (!pr_visit_block<UNR>(stage[wid], sbox[wid], T, BL, BH, CBL, blk, nx, ny, nz, valid, inf, best, bchunk, tie, chunks))
            continue;   // no lane's own box test passed: every minimum (and so thr) is unchanged
        ++scanned;
        thr = pr_ord2f(__reduce_max_sync(0xffffffffu, valid ? pr_f2ord(best) : (int)0x80000000));
    }
    // ---- the lowest original index at the minimum: inside the winning chunk ... ----
    int bidx = 0x7fffffff;
    {
        const float4 *tc = T + bchunk * 8;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 t = __ldg(tc + i);
            const float d = sqdist_ref(q.x, q.y, q.z, t.x, t.y, t.z);
            if (d == best) bidx = min(bidx, __float_as_int(t.w));
        }
    }
    // ---- ... and, for a lane that met its minimum in two chunks, over every block that could hold it ----
    const unsigned ties = __ballot_sync(0xffffffffu, tie && valid);
    if (ties != 0u) {
        for (int blk = 0; blk < nblk; ++blk) {
            const float s = pr_box_d2(glo[0], glo[1], glo[2], ghi[0], ghi[1], ghi[2], __ldg(BL + blk), __ldg(BH + blk));
            if (!(s <= thr)) continue;   // warp-uniform
            const float4 *tb = T + blk * PR_BLOCK;
            for (int i = 0; i < PR_BLOCK; ++i) {
                const float4 t = __ldg(tb + i);
                const float d = sqdist_ref(q.x, q.y, q.z, t.x, t.y, t.z);
                if (tie && d == best) bidx = min(bidx, __float_as_int(t.w));
            }
        }
    }
    if (valid) p.out[(size_t)b * p.nq + __float_as_int(q.w)] = pack_dist_idx(best, bidx);
    if (p.stats != nullptr && lane == 0) {
        atomicAdd(p.stats + 0, scanned);
        if (ties != 0u) atomicAdd(p.stats + 1, 1u);
        atomicAdd(p.stats + 2, 1u);
        atomicAdd(p.stats + 3, chunks);
    }
}

// CTAs of one direction in nn_prune_kernel: eight query groups per CTA
static inline int pr_ctas(const PruneParams &q) {
    const int groups = (q.nq + PR_GROUP - 1) / PR_GROUP;
    return q.B * ((groups + PR_THREADS / 32 - 1) / (PR_THREADS / 32));
}
// Both directions of a cloud pair: the one with fewer queries (longer chains per group: more target blocks) goes first
static inline PrunePair pr_pair(const PruneParams &a, const PruneParams &b) {
    PrunePair pp = {};
    const bool a_first = a.nq <= b.nq;
    pp.d[0] = a_first ? a : b, pp.d[1] = a_first ? b : a;
    pp.ctas0 = pr_ctas(pp.d[0]);
    return pp;
}
// nn_prune_kernel over the pair: pp.ctas0 CTAs for d[0] (0: d[0] is launched elsewhere), then d[1]'s; a programmatic dependent
// of the sort queued before it
static inline void pr_launch(const PrunePair &pp, cudaStream_t stream) {
    const unsigned grid = (unsigned)(pp.ctas0 + pr_ctas(pp.d[1]));
    const int nt = pp.ctas0 == 0 || pp.d[1].nt > pp.d[0].nt ? pp.d[1].nt : pp.d[0].nt;
    pr_rows(pr_nblk(nt), [&](auto r) { launch_pdl(nn_prune_kernel<decltype(r)::value>, dim3(grid), dim3(PR_THREADS), stream, pp); });
}

// Cooperative form for a direction with FEW query groups and many target blocks (C2: 2048 groups against 256 blocks each): one
// CTA per group, each of its eight warps walks an eighth of the blocks nearest first; the running minima are shared through
// shared-memory atomics, so every warp stops where a single warp would (its bound is never below the final one: no block that
// matters is skipped), and warp 0 merges the eight partial results.  A group's dependent chain -- up to 256
// block visits of 0.35 us in one warp, which set the duration of the whole launch (118 us on one batch of the bench's generator,
// 167 us on others with the same instruction count) -- becomes an eighth as long.  Launched on a side stream next to the other
// direction's nn_prune_kernel.
template <int BOXR>
__global__ void __launch_bounds__(PR_THREADS) nn_prune_coop_kernel(const PruneParams p) {
    __shared__ __align__(16) float stage[PR_THREADS / 32][3][PR_BLOCK];
    __shared__ float4 sbox[PR_THREADS / 32][16];
    __shared__ unsigned s_best[PR_GROUP];                      // running minimum per query over all warps (float bits, >= 0)
    __shared__ float m_best[PR_THREADS / 32][PR_GROUP];
    __shared__ int m_chunk[PR_THREADS / 32][PR_GROUP], m_tie[PR_THREADS / 32][PR_GROUP];
    if (p.select != nullptr && *p.select != 0) return;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int groups = (p.nq + PR_GROUP - 1) / PR_GROUP;
    const int b = (int)blockIdx.x / groups;
    const int g = (int)blockIdx.x % groups;
    if (wid == 0) s_best[lane] = 0x7f800000u;
    __syncthreads();
    const int nblk = pr_nblk(p.nt);
    const int bt = p.tdiv > 1 ? b / p.tdiv : b, bq = p.qdiv > 1 ? b / p.qdiv : b;
    const float4 *T = p.t + (size_t)bt * pr_npad(p.nt);
    const float4 *BL = p.tbox + (size_t)bt * 2 * nblk, *BH = BL + nblk;
    const int nchunk = pr_npad(p.nt) / 8;   // lanes 0-7 / 8-15 stage the lower / upper corners of a block's eight chunk boxes
    const float4 *CBL = p.tcbox + (size_t)bt * 2 * nchunk + (lane >> 3) * nchunk + (lane & 7);
    const float inf = __int_as_float(0x7f800000);
    const int qi = g * PR_GROUP + lane;
    const bool valid = qi < p.nq;
    const float4 q = p.q[(size_t)bq * pr_npad(p.nq) + qi];   // the padding records are NaN: they never win, nothing is stored
    // ---- the group's box ----
    float glo[3], ghi[3];
    {
        const float v[3] = {q.x, q.y, q.z};
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            // NaN (padding) must not take part: +inf / -inf are neutral
            const float a = valid ? v[c] : inf, z = valid ? v[c] : -inf;
            glo[c] = pr_ord2f(__reduce_min_sync(0xffffffffu, pr_f2ord(a)));
            ghi[c] = pr_ord2f(__reduce_max_sync(0xffffffffu, pr_f2ord(z)));
        }
    }
    // ---- squared box-to-box distances, scaled down (see the header) ----
    // warp w owns the blocks w, w + 8, w + 16, ... (consecutive Hilbert blocks are neighbours: every warp gets an even sample
    // of the cloud) and runs the nearest-first walk over ITS blocks only -- no selection work is repeated
    constexpr int WARPS = PR_THREADS / 32;
    constexpr int CBOXR = (BOXR + WARPS - 1) / WARPS;
    float bd[CBOXR];
#pragma unroll
    for (int r = 0; r < CBOXR; ++r) {
        const int blk = wid + WARPS * (r * 32 + lane);
        bd[r] = inf;
        if (blk < nblk) bd[r] = pr_box_d2(glo[0], glo[1], glo[2], ghi[0], ghi[1], ghi[2], __ldg(BL + blk), __ldg(BH + blk));
    }
    const float2 nx = make_float2(-q.x, -q.x), ny = make_float2(-q.y, -q.y), nz = make_float2(-q.z, -q.z);
    float best = inf;
    int bchunk = 0;
    bool tie = false;
    float thr = inf;   // the largest running minimum of the group's lanes
    unsigned scanned = 0, chunks = 0;
    for (;;) {
        unsigned key = 0xffffffffu;   // (distance bits without the low 9, slot = r * 32 + lane of the owned block)
#pragma unroll
        for (int r = 0; r < CBOXR; ++r) key = min(key, (__float_as_uint(bd[r]) & 0xfffffe00u) | (unsigned)(r * 32 + lane));
        key = __reduce_min_sync(0xffffffffu, key);
        // the bound uses what ANY warp has found so far for each query (a real distance to that query: never below its minimum)
        const float cap = __uint_as_float(*(volatile unsigned *)&s_best[lane]);
        thr = pr_ord2f(__reduce_max_sync(0xffffffffu, valid ? pr_f2ord(fminf(best, cap)) : (int)0x80000000));
        if (key >= 0x7f800000u || !(__uint_as_float(key & 0xfffffe00u) <= thr)) break;
        const int slot = (int)(key & 0x1ffu);
#pragma unroll
        for (int r = 0; r < CBOXR; ++r)
            if (r * 32 + lane == slot) bd[r] = inf;
        if (!pr_visit_block<PR_UNROLL>(stage[wid], sbox[wid], T, BL, BH, CBL, wid + WARPS * slot, nx, ny, nz, valid, cap, best, bchunk,
                                       tie, chunks))
            continue;
        ++scanned;
        if (valid) atomicMin(&s_best[lane], __float_as_uint(best));
    }
    // ---- merge the eight warps' results (warp 0 finishes the group) ----
    m_best[wid][lane] = best, m_chunk[wid][lane] = bchunk, m_tie[wid][lane] = tie ? 1 : 0;
    if (p.stats != nullptr && lane == 0 && wid != 0) atomicAdd(p.stats + 0, scanned), atomicAdd(p.stats + 3, chunks);
    __syncthreads();
    if (wid != 0) return;
#pragma unroll
    for (int w = 1; w < PR_THREADS / 32; ++w) {
        const float mb = m_best[w][lane];
        const int mc = m_chunk[w][lane];
        const bool mt = m_tie[w][lane] != 0;
        if (mb < best) {
            best = mb, bchunk = mc, tie = mt;
        } else if (mb == best && mb < inf) {
            tie = tie || mt || mc != bchunk;
        }
    }
    thr = pr_ord2f(__reduce_max_sync(0xffffffffu, valid ? pr_f2ord(best) : (int)0x80000000));
    // ---- the lowest original index at the minimum: inside the winning chunk ... ----
    int bidx = 0x7fffffff;
    {
        const float4 *tc = T + bchunk * 8;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 t = __ldg(tc + i);
            const float d = sqdist_ref(q.x, q.y, q.z, t.x, t.y, t.z);
            if (d == best) bidx = min(bidx, __float_as_int(t.w));
        }
    }
    // ---- ... and, for a lane that met its minimum in two chunks, over every block that could hold it ----
    const unsigned ties = __ballot_sync(0xffffffffu, tie && valid);
    if (ties != 0u) {
        for (int blk = 0; blk < nblk; ++blk) {
            const float s = pr_box_d2(glo[0], glo[1], glo[2], ghi[0], ghi[1], ghi[2], __ldg(BL + blk), __ldg(BH + blk));
            if (!(s <= thr)) continue;   // warp-uniform
            const float4 *tb = T + blk * PR_BLOCK;
            for (int i = 0; i < PR_BLOCK; ++i) {
                const float4 t = __ldg(tb + i);
                const float d = sqdist_ref(q.x, q.y, q.z, t.x, t.y, t.z);
                if (tie && d == best) bidx = min(bidx, __float_as_int(t.w));
            }
        }
    }
    if (valid) p.out[(size_t)b * p.nq + __float_as_int(q.w)] = pack_dist_idx(best, bidx);
    if (p.stats != nullptr && lane == 0) {
        atomicAdd(p.stats + 0, scanned);
        if (ties != 0u) atomicAdd(p.stats + 1, 1u);
        atomicAdd(p.stats + 2, 1u);
        atomicAdd(p.stats + 3, chunks);
    }
}

}  // namespace genpc
