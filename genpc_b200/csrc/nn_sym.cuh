// nn_sym.cuh -- symmetric Chamfer scan: every distance is evaluated ONCE and feeds both directions.
//
// d(j,k) = fma(dz,dz,fma(dx,dx,dy*dy)) is bit-identical whichever cloud plays "query" (the differences only
// change sign and every product is a square), so the N x M matrix the reference evaluates twice
// (chamfer3D.cu:142-143) is evaluated once here: the FMA pipe -- the unit that bounds this kernel (2 packed
// instructions/clk/SM, 3 per point pair) -- does half the work per directed pair.
//
//   rows  = the cloud held in registers (QT points per thread, a warp owns 32*QT CONSECUTIVE rows),
//   cols  = the cloud swept through shared memory in spans (SoA, NaN padded), 32 columns per block.
//   row side: running minimum by FMNMX3, winning 8-column chunk id tracked, exact lowest index recovered by a
//             re-scan of that chunk, merged across column spans by a packed 64-bit atomicMin (as nn_core.cuh);
//   col side: per 32-column block every lane folds its QT rows into 32 accumulators (FMNMX3 over row pairs),
//             one warp reduction per column (REDUX.MIN) leaves lane l with the warp-wide minimum of column l, and ONE
//             coalesced 64-bit atomicMin per lane publishes (dist_bits << 32 | row_block_id).  The exact lowest
//             row index is recovered afterwards by nn_sym_epilogue_kernel, which re-scans only the winning
//             32*QT-row block of each column (lowest block wins ties, first match inside it => lowest index).
#pragma once
#include "nn_core.cuh"

namespace genpc {

constexpr int SYM_THREADS = 256;
constexpr int SYM_SPAN_MAX = 1024;  // columns staged per item (12 B of shared memory each)
#ifndef GENPC_SYM_CHUNK
#define GENPC_SYM_CHUNK 8
#endif
constexpr int SYM_CHUNK = GENPC_SYM_CHUNK;  // row-side index-recovery granularity (columns)

struct SymParams {
    const float *rows;             // [B][nr][3]
    const float *cols;             // [B][nc][3]
    unsigned long long *prow;      // [B][nr]  (dist, col index)
    unsigned long long *pcol;      // [B][nc]  (dist, row block id)
    int nr, nc, rtiles, cspans, span;
    int rblock_base;               // added to published row-block ids (row shard offset / rows_per_block)
    // host-fed launches (genpc_chamfer_forward_host): cloud pair b may be read once gate[b / gate_pairs] has reached
    // gate_gen -- the H2D copy of its chunk has landed (written by a 4-byte DMA queued behind the chunk's copies)
    const unsigned *gate;
    unsigned gate_gen;
    int gate_pairs;
    // selection flag of the pruned scans (nn_prune.cuh, nn_grid.cuh): when set, this launch only runs if *select != 0, i.e.
    // the sort's range check or the grid probe handed the work back to the exhaustive kernels; nullptr: always run
    const int *select;
    // ragged batches (genpc_chamfer_forward_ragged): points of each row / column cloud [B], the rest of its nr / nc stride is
    // padding that is never read; nullptr: every cloud fills its stride
    // (nn_sym_kernel only: the balanced form cuts its units by the strides, not by the real work, and carrying the row length
    // into it cost it 12-16 more bytes of spills)
    const int *len_r, *len_c;
};

// points of cloud b of a ragged batch, clamped to [0, stride] so that no index leaves the cloud whatever a caller passes
__device__ __forceinline__ int sym_len(const int *len, int b, int stride) {
    return len == nullptr ? stride : min(max(__ldg(len + b), 0), stride);
}

// Work items of the symmetric scan over B cloud pairs: row tiles of SYM_THREADS * QT rows x column spans, the span the largest
// that still gives >= 2 waves of work items (3 CTAs x SMs), at least 256 columns.  Returns B * rtiles * cspans.
static inline long long sym_tiling(int B, int nr, int nc, int QT, int &rtiles, int &span, int &cspans) {
    rtiles = (nr + SYM_THREADS * QT - 1) / (SYM_THREADS * QT);
    span = SYM_SPAN_MAX;
    const long long want = 2LL * 3 * GENPC_NUM_SMS;
    while (span > 256 && (long long)B * rtiles * ((nc + span - 1) / span) < want) span >>= 1;
    cspans = (nc + span - 1) / span;
    return (long long)B * rtiles * cspans;
}

// Coordinates arriving by DMA while the kernel is resident must not go through the non-coherent path (ld.global.nc
// assumes data that is read-only for the whole launch): gated launches read them with ld.global.cg instead.
template <bool COHERENT>
__device__ __forceinline__ float ld_coord(const float *p) {
    return COHERENT ? __ldcg(p) : __ldg(p);
}

// One work item: row tile `rt` (SYM_THREADS*QT rows) x column span [c0, c0+span) of ONE cloud pair.
// rows/cols/prow/pcol point at the first element of the pair's clouds / packed words.  colT: optional similarity
// applied to the columns while they are staged (registration: the moving cloud), nullptr = identity.
// nr_pub >= nr >= 1 (ragged batch: nr is the row cloud's length, nr_pub its stride): rows [nr, nr_pub) are not read -- they
// hold NaN like the rows past the cloud, so they never win a column -- but publish into their own (padding) packed words, which
// nobody reads and the fused epilogue re-arms.  (Bounding the loads themselves by the length, or the publishing, cost
// nn_sym_kernel<4> 12 more bytes of spills: ptxas -v.)
template <int QT, bool COHERENT = false>
__device__ __forceinline__ void nn_sym_item(float (*s)[SYM_SPAN_MAX], const float *__restrict__ rows, int nr, int rt,
                                            const float *__restrict__ cols, int nc, int c0, int span,
                                            const Similarity *colT, unsigned long long *__restrict__ prow_,
                                            unsigned long long *__restrict__ pcol_, int rblock_base = 0, int nr_pub = -1) {
    if (nr_pub < 0) nr_pub = nr;
    static_assert(QT % 2 == 0, "rows are folded in pairs");
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cnt = min(span, nc - c0);
    const int cnt32 = (cnt + 31) & ~31;
    const float qnan = __int_as_float(0x7fc00000);
    // ---- stage the column span ----
    const float *cp = cols + (size_t)c0 * 3;
    for (int k = tid; k < cnt32; k += SYM_THREADS) {
        float x = qnan, y = qnan, z = qnan;
        if (k < cnt) {
            x = ld_coord<COHERENT>(cp + k * 3), y = ld_coord<COHERENT>(cp + k * 3 + 1), z = ld_coord<COHERENT>(cp + k * 3 + 2);
            if (colT != nullptr) apply_similarity(*colT, x, y, z);
        }
        s[0][k] = x, s[1][k] = y, s[2][k] = z;
    }
    // ---- rows into registers (negated; NaN for out-of-range rows: they never win a min on either side) ----
    float2 nqx[QT], nqy[QT], nqz[QT];
    float best[QT];
    int bchunk[QT];
    const int rblock = rt * (SYM_THREADS / 32) + warp;          // global id of this warp's 32*QT-row block
    const int jbase = rblock * (32 * QT) + lane;
    const float *rp = rows;
#pragma unroll
    for (int qi = 0; qi < QT; ++qi) {
        const int j = jbase + qi * 32;
        float x = qnan, y = qnan, z = qnan;
        if (j < nr_pub) {   // (rows [nr, nr_pub): a real row is loaded and replaced by NaN -- see above)
            const int jr = min(j, nr - 1);
            x = ld_coord<COHERENT>(rp + (size_t)jr * 3), y = ld_coord<COHERENT>(rp + (size_t)jr * 3 + 1),
            z = ld_coord<COHERENT>(rp + (size_t)jr * 3 + 2);
            if (j >= nr) x = y = z = qnan;
        }
        nqx[qi] = make_float2(-x, -x);
        nqy[qi] = make_float2(-y, -y);
        nqz[qi] = make_float2(-z, -z);
        best[qi] = __int_as_float(0x7f800000);
        bchunk[qi] = 0;
    }
    __syncthreads();

    const float4 *sx4 = reinterpret_cast<const float4 *>(s[0]);
    const float4 *sy4 = reinterpret_cast<const float4 *>(s[1]);
    const float4 *sz4 = reinterpret_cast<const float4 *>(s[2]);
    unsigned long long *pcol = pcol_ + c0;
    const float inf = __int_as_float(0x7f800000);
    for (int blk = 0; blk < cnt32 / 32; ++blk) {
        float cacc[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) cacc[i] = inf;
#pragma unroll
        for (int sub = 0; sub < 32 / SYM_CHUNK; ++sub) {
            float cm[QT];
#pragma unroll
            for (int qi = 0; qi < QT; ++qi) cm[qi] = inf;
#pragma unroll
            for (int kk = 0; kk < SYM_CHUNK / 4; ++kk) {
                const int g = blk * 8 + sub * (SYM_CHUNK / 4) + kk;  // float4 group index
                const float4 X = sx4[g], Y = sy4[g], Z = sz4[g];
                const int t = sub * SYM_CHUNK + kk * 4;               // column offset inside the block
#pragma unroll
                for (int qi = 0; qi < QT; qi += 2) {
                    const float2 a0 = sqdist_ref_x2(nqx[qi], nqy[qi], nqz[qi], make_float2(X.x, X.y),
                                                    make_float2(Y.x, Y.y), make_float2(Z.x, Z.y));
                    const float2 e0 = sqdist_ref_x2(nqx[qi], nqy[qi], nqz[qi], make_float2(X.z, X.w),
                                                    make_float2(Y.z, Y.w), make_float2(Z.z, Z.w));
                    const float2 a1 = sqdist_ref_x2(nqx[qi + 1], nqy[qi + 1], nqz[qi + 1], make_float2(X.x, X.y),
                                                    make_float2(Y.x, Y.y), make_float2(Z.x, Z.y));
                    const float2 e1 = sqdist_ref_x2(nqx[qi + 1], nqy[qi + 1], nqz[qi + 1], make_float2(X.z, X.w),
                                                    make_float2(Y.z, Y.w), make_float2(Z.z, Z.w));
                    cm[qi] = fmin3(cm[qi], a0.x, a0.y);
                    cm[qi] = fmin3(cm[qi], e0.x, e0.y);
                    cm[qi + 1] = fmin3(cm[qi + 1], a1.x, a1.y);
                    cm[qi + 1] = fmin3(cm[qi + 1], e1.x, e1.y);
                    cacc[t + 0] = fmin3(cacc[t + 0], a0.x, a1.x);
                    cacc[t + 1] = fmin3(cacc[t + 1], a0.y, a1.y);
                    cacc[t + 2] = fmin3(cacc[t + 2], e0.x, e1.x);
                    cacc[t + 3] = fmin3(cacc[t + 3], e0.y, e1.y);
                }
            }
#pragma unroll
            for (int qi = 0; qi < QT; ++qi) {
                if (cm[qi] < best[qi]) {  // strict: the earliest chunk keeps ties
                    best[qi] = cm[qi];
                    bchunk[qi] = blk * (32 / SYM_CHUNK) + sub;
                }
            }
        }
        // ---- column side: warp-wide minimum of column (blk*32 + lane), published with the row-block id ----
        unsigned mine = 0x7f800000u;  // distances are >= 0: their bit patterns order like the floats
#pragma unroll
        for (int c = 0; c < 32; ++c) {
            const unsigned r = __reduce_min_sync(0xffffffffu, __float_as_uint(cacc[c]));
            if (lane == c) mine = r;
        }
        const float cmin = __uint_as_float(mine);
        // every in-range column publishes, also when its minimum is +inf (NaN / overflowing coordinates): no packed word
        // is ever left unarmed, so the epilogue and the gradient kernels always see an in-range block / index
        const int col = blk * 32 + lane;
        if (col < cnt) atomicMin(pcol + col, pack_dist_idx(cmin, rblock_base + rblock));
    }

    // ---- row side: exact lowest column index inside the winning chunk, merged across column spans ----
    unsigned long long *prow = prow_;
#pragma unroll
    for (int qi = 0; qi < QT; ++qi) {
        const int j = jbase + qi * 32;
        if (j >= nr_pub) continue;
        // every in-range row publishes, also when its minimum stayed +inf (NaN / overflowing coordinates: the re-scan finds
        // no match and reports the first column of the span, like nn_scan_item) -- no packed word is ever left unarmed
        const float qx = -nqx[qi].x, qy = -nqy[qi].x, qz = -nqz[qi].x;
        const int cb = bchunk[qi] * SYM_CHUNK;
        int kbest = 0;
#pragma unroll
        for (int k = SYM_CHUNK - 1; k >= 0; --k) {
            const float dd = sqdist_ref(qx, qy, qz, s[0][cb + k], s[1][cb + k], s[2][cb + k]);
            if (dd == best[qi]) kbest = k;
        }
        atomicMin(prow + j, pack_dist_idx(best[qi], c0 + cb + kbest));
    }
}

template <int QT>
__global__ void __launch_bounds__(SYM_THREADS, 2) nn_sym_kernel(const SymParams p) {
    __shared__ __align__(16) float s[3][SYM_SPAN_MAX];
    cudaGridDependencySynchronize();   // a programmatic dependent of the pruned scan when it is that scan's fall-back
    cudaTriggerProgrammaticLaunchCompletion();
    if (p.select != nullptr && *p.select == 0) return;
    int item = blockIdx.x;
    const int cs = item % p.cspans;
    item /= p.cspans;
    const int rt = item % p.rtiles;
    const int b = item / p.rtiles;
    // a ragged batch's grid is sized by the strides: an item whose row tile or column span lies wholly in the pair's padding
    // has nothing to do (CTA-uniform)
    const int nr = sym_len(p.len_r, b, p.nr), nc = sym_len(p.len_c, b, p.nc);
    if (rt * (SYM_THREADS * QT) >= nr || cs * p.span >= nc) return;
    nn_sym_item<QT>(s, p.rows + (size_t)b * p.nr * 3, nr, rt, p.cols + (size_t)b * p.nc * 3, nc, cs * p.span, p.span,
                    nullptr, p.prow + (size_t)b * p.nr, p.pcol + (size_t)b * p.nc, p.rblock_base, p.nr);
}

// Host-fed form: same work items, but the clouds are still arriving from pinned host memory while the kernel runs.
// Thread 0 of every CTA waits (acquire, system scope) until the generation word of its cloud pair's chunk has been
// written by the copy stream, then the CTA proceeds exactly like nn_sym_kernel.  CTAs are dispatched in blockIdx
// order == batch order == copy order, so waiting CTAs only ever wait for the chunk the copy engine is working on.
// A spin that outlives GATE_TIMEOUT_CLK raises gate[GATE_ERR_SLOT] and goes on (garbage out, reported by the host call
// of the NEXT step) rather than hanging the GPU.
constexpr int GATE_MAX_CHUNKS = 64;
constexpr int GATE_ERR_SLOT = GATE_MAX_CHUNKS;
constexpr long long GATE_TIMEOUT_CLK = 4000000000LL;  // ~2 s at 1.965 GHz

template <int QT>
__global__ void __launch_bounds__(SYM_THREADS, 2) nn_sym_gated_kernel(const SymParams p) {
    __shared__ __align__(16) float s[3][SYM_SPAN_MAX];
    cudaTriggerProgrammaticLaunchCompletion();   // (never launched as a dependent: it follows memsets)
    if (p.select != nullptr && *p.select == 0) return;
    int item = blockIdx.x;
    const int cs = item % p.cspans;
    item /= p.cspans;
    const int rt = item % p.rtiles;
    const int b = item / p.rtiles;
    if (threadIdx.x == 0) {
        const unsigned *g = p.gate + b / p.gate_pairs;
        const long long t0 = clock64();
        for (;;) {
            unsigned v;
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(g) : "memory");
            if ((int)(v - p.gate_gen) >= 0) break;
            if (clock64() - t0 > GATE_TIMEOUT_CLK) {
                atomicExch(const_cast<unsigned *>(p.gate) + GATE_ERR_SLOT, 1u);
                break;
            }
            __nanosleep(128);
        }
    }
    __syncthreads();
    nn_sym_item<QT, true>(s, p.rows + (size_t)b * p.nr * 3, p.nr, rt, p.cols + (size_t)b * p.nc * 3, p.nc, cs * p.span,
                          p.span, nullptr, p.prow + (size_t)b * p.nr, p.pcol + (size_t)b * p.nc, p.rblock_base);
}

// Balanced form ("stream-K" over the distance matrix): the work of the whole launch is counted in UNITS of one row
// tile x one 32-column block, linearised as (cloud pair, row tile, column block), and cut into gridDim.x equal
// contiguous ranges -- one per resident CTA (2 per SM).  A CTA walks its range as a sequence of ordinary work items
// (same row tile, up to SYM_SPAN_MAX consecutive columns), so every CTA executes the same number of column blocks
// +-1 whatever the problem shape: no partial last wave (C2: 1024 items over 296 slots = 3.46 waves before) and
// B = 1 problems fill the machine.  Results are merged by the same packed atomicMin words, hence bit-identical.
template <int QT>
__global__ void __launch_bounds__(SYM_THREADS, 2) nn_sym_balanced_kernel(const SymParams p, int total_units,
                                                                          int units_per_job) {
    __shared__ __align__(16) float s[3][SYM_SPAN_MAX];
    cudaGridDependencySynchronize();   // a programmatic dependent of the pruned scan when it is that scan's fall-back
    cudaTriggerProgrammaticLaunchCompletion();
    if (p.select != nullptr && *p.select == 0) return;
    int u = (int)((long long)total_units * blockIdx.x / gridDim.x);
    const int u_end = (int)((long long)total_units * (blockIdx.x + 1) / gridDim.x);
    int job = u / units_per_job;
    int blk = u - job * units_per_job;
    while (u < u_end) {
        int nblk = min(min(units_per_job - blk, SYM_SPAN_MAX / 32), u_end - u);  // row tile end / one smem span / range end
        const int rt = job % p.rtiles, b = job / p.rtiles;
        nn_sym_item<QT>(s, p.rows + (size_t)b * p.nr * 3, p.nr, rt, p.cols + (size_t)b * p.nc * 3, p.nc, blk * 32, nblk * 32,
                        nullptr, p.prow + (size_t)b * p.nr, p.pcol + (size_t)b * p.nc, p.rblock_base);
        u += nblk, blk += nblk;
        if (blk == units_per_job) blk = 0, ++job;
        __syncthreads();  // every warp is done with the span before the next item overwrites it
    }
}

// Exact lowest row index of one column from its published (dist, row block) word: the calling WARP re-scans the
// winning block (32*NS consecutive rows) for the first row whose distance equals dist.  All NS strips are loaded
// up front (one exposed memory latency instead of one per strip; the scan is latency bound, not bandwidth bound).
template <int NS>
__device__ __forceinline__ int sym_fix_column_t(const float *__restrict__ rp, int nr, float cx, float cy, float cz, float d,
                                                int blk, int lane) {
    float rx[NS], ry[NS], rz[NS];
    const int r0 = blk * (32 * NS);
#pragma unroll
    for (int q = 0; q < NS; ++q) {
        const int j = min(r0 + q * 32 + lane, nr - 1);
        rx[q] = __ldg(rp + (size_t)j * 3), ry[q] = __ldg(rp + (size_t)j * 3 + 1), rz[q] = __ldg(rp + (size_t)j * 3 + 2);
    }
    int found = 0;
    bool done = false;
#pragma unroll
    for (int q = 0; q < NS; ++q) {
        const int j = r0 + q * 32 + lane;
        const bool hit = (j < nr) && (sqdist_ref(cx, cy, cz, rx[q], ry[q], rz[q]) == d);
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if (!done && m) {
            found = r0 + q * 32 + __ffs(m) - 1;
            done = true;
        }
    }
    return found;
}

// 128-row block, vector form: the block is 1536 contiguous bytes, every lane takes 48 of them (rows r0 + 4*lane .. +3)
// with three LDG.128 instead of twelve LDG.32 -- the fix-up is bound by load instructions and their latency, not by
// bytes.  Needs the block entirely inside the cloud and a 16-byte aligned block start; the caller checks both.
__device__ __forceinline__ int sym_fix_column_v4(const float *__restrict__ rp, float cx, float cy, float cz, float d, int blk,
                                                 int lane) {
    const int r0 = blk * 128;
    const float4 *bp = reinterpret_cast<const float4 *>(rp + (size_t)r0 * 3) + lane * 3;
    const float4 v0 = __ldg(bp), v1 = __ldg(bp + 1), v2 = __ldg(bp + 2);
    int first = 4;  // lowest matching row of this lane's four, 4 = none (tested last to first)
    if (sqdist_ref(cx, cy, cz, v2.y, v2.z, v2.w) == d) first = 3;
    if (sqdist_ref(cx, cy, cz, v1.z, v1.w, v2.x) == d) first = 2;
    if (sqdist_ref(cx, cy, cz, v0.w, v1.x, v1.y) == d) first = 1;
    if (sqdist_ref(cx, cy, cz, v0.x, v0.y, v0.z) == d) first = 0;
    const unsigned m = __ballot_sync(0xffffffffu, first < 4);
    if (m == 0) return 0;
    const int src = __ffs(m) - 1;  // lanes hold ascending rows: the lowest lane with a match holds the lowest index
    return r0 + 4 * src + __shfl_sync(0xffffffffu, first, src);
}

__device__ __forceinline__ int sym_fix_column(const float *__restrict__ rp, int nr, int rows_per_block, float cx, float cy,
                                              float cz, float d, int blk, int lane) {
    if (rows_per_block == 128) {
        if ((blk + 1) * 128 <= nr && (reinterpret_cast<size_t>(rp) & 15) == 0)  // warp-uniform
            return sym_fix_column_v4(rp, cx, cy, cz, d, blk, lane);
        return sym_fix_column_t<4>(rp, nr, cx, cy, cz, d, blk, lane);
    }
    if (rows_per_block == 64) return sym_fix_column_t<2>(rp, nr, cx, cy, cz, d, blk, lane);
    int found = 0;  // generic: any other block height
    for (int r0 = blk * rows_per_block; r0 < (blk + 1) * rows_per_block; r0 += 32) {
        const int j = r0 + lane;
        bool hit = false;
        if (j < nr) {
            const float dd = sqdist_ref(cx, cy, cz, __ldg(rp + (size_t)j * 3), __ldg(rp + (size_t)j * 3 + 1),
                                        __ldg(rp + (size_t)j * 3 + 2));
            hit = (dd == d);
        }
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if (m) {
            found = r0 + __ffs(m) - 1;
            break;
        }
    }
    return found;
}

// Optional extra duties of the forward epilogue (genpc_chamfer_forward_fused): everything that used to be separate tiny
// launches around the scan in a loss step -- the loss reduction, the zero-fill of the gradient accumulators that the
// backward kernel adds into, and re-arming the packed words so that the next call on the same workspace needs no memset.
struct EpiFuse {
    double *partial;        // one slot per epilogue CTA; nullptr: no loss
    unsigned *ticket;       // zero between launches (re-armed by the last CTA)
    float *loss_out;        // device scalar
    double fcol, frow;      // loss = fcol * sum_cols f(d) + frow * sum_rows f(d)   (w / count; 0 drops the side);
                            // ragged batch: each term is f(d) / len[b] and fcol / frow are w / B
    int use_sqrt;           // f = sqrt or identity
    int rearm;              // store all-ones back into every packed word after reading it
    float *zero[2];         // buffers to zero-fill, or nullptr
    size_t nzero[2];        // their sizes in floats
    const unsigned *err_flag;  // host-fed launches: the feed's error word -- a timed-out gate poisons the loss with NaN
    const int *select;         // selection flag of the pruned scans: *select == 0 -> the column words already hold exact indices
    // ragged batch (SymParams::len_r / len_c; nullptr: full strides): a row or column past its cloud's length, or of a pair whose
    // other cloud is empty, has no neighbour -- it gets dist 0, idx -1 and no loss term; the fix-up stops at the row length
    const int *len_r, *len_c;
};

__device__ __forceinline__ void epi_zero_fill(float *z, size_t n, size_t g, size_t total_threads) {
    if (z == nullptr) return;
    if ((reinterpret_cast<size_t>(z) & 15) == 0) {
        float4 *z4 = reinterpret_cast<float4 *>(z);
        const size_t n4 = n >> 2;
        for (size_t i = g; i < n4; i += total_threads) z4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (g < (n & 3)) z[(n4 << 2) + g] = 0.f;
    } else {
        for (size_t i = g; i < n; i += total_threads) z[i] = 0.f;
    }
}

// Forward epilogue in ONE launch: blocks [0, fix_blocks) resolve the column words (exact lowest row index from the
// winning row block) and write dist/idx of the column cloud; the remaining blocks unpack the row words into dist/idx of
// the row cloud.  CTAs are FAT -- a warp resolves EPI_CPW consecutive columns (lane k fetches word + point of column k up
// front, the columns are handed round by shuffles and their row-block loads are independent), a thread unpacks EPI_RPT
// rows -- because the thin form (one column per warp, one row per thread: 10 240 CTAs on C2) is bound by the dependent
// L2 latencies of every CTA, not by bytes.  FUSED: additionally the duties of EpiFuse; the loss is deterministic (one
// double partial per CTA from a fixed tree, the last CTA -- ticket -- adds the partials of each side in index order).
constexpr int EPI_CPW = 8;                        // columns per warp
constexpr int EPI_COLS_PER_CTA = 8 * EPI_CPW;     // 256 threads
constexpr int EPI_RPT = 8;                        // rows per thread
constexpr int EPI_ROWS_PER_CTA = 256 * EPI_RPT;

template <bool FUSED>
static __global__ void __launch_bounds__(256) nn_sym_epilogue_kernel(const float *__restrict__ rows, const float *__restrict__ cols,
                                                                     unsigned long long *__restrict__ prow,
                                                                     unsigned long long *__restrict__ pcol, int B, int nr,
                                                                     int nc, int rows_per_block, unsigned fix_blocks,
                                                                     float *__restrict__ dist_r, int *__restrict__ idx_r,
                                                                     float *__restrict__ dist_c, int *__restrict__ idx_c,
                                                                     const EpiFuse f) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // a programmatic dependent of the scan: the packed words, the selection flag, the outputs and the gradient accumulators are
    // all touched below this point
    cudaGridDependencySynchronize();
    const bool cols_exact = f.select != nullptr && *f.select == 0;   // a pruned scan ran: nothing to fix up (warp-uniform)
    double term = 0.0;  // sum of f(d) over the output elements this thread owns
    if (blockIdx.x >= fix_blocks) {
        const size_t n = (size_t)B * nr;
        const size_t i0 = (size_t)(blockIdx.x - fix_blocks) * EPI_ROWS_PER_CTA + threadIdx.x;
        if (f.len_r != nullptr) {
            // ragged batch, one row at a time (a division per row in the unrolled form below raised the registers of every
            // epilogue launch from 32 / 47 to 64): a row past its cloud's length, or of a pair whose column cloud is empty, has no
            // neighbour; the loss term of a row is f(d) / (its cloud's length)
#pragma unroll 1
            for (int k = 0; k < EPI_RPT; ++k) {
                const size_t i = i0 + (size_t)k * 256;
                if (i >= n) break;
                const int b = (int)(i / (size_t)nr), len = sym_len(f.len_r, b, nr);
                const bool has_nn = (int)(i - (size_t)b * nr) < len && sym_len(f.len_c, b, nc) > 0;
                const unsigned long long w = __ldcg(prow + i);
                const float d = has_nn ? __uint_as_float((unsigned)(w >> 32)) : 0.f;
                dist_r[i] = d;
                idx_r[i] = has_nn ? (int)(unsigned)(w & 0xffffffffu) : -1;
                if (FUSED) {
                    if (f.rearm) prow[i] = ~0ull;
                    if (has_nn) term += (double)(f.use_sqrt ? __fsqrt_rn(d) : d) / (double)len;
                }
            }
        } else {
            unsigned long long w[EPI_RPT];
#pragma unroll
            for (int k = 0; k < EPI_RPT; ++k) {
                const size_t i = i0 + (size_t)k * 256;
                w[k] = (i < n) ? __ldcg(prow + i) : 0ull;
            }
#pragma unroll
            for (int k = 0; k < EPI_RPT; ++k) {
                const size_t i = i0 + (size_t)k * 256;
                if (i < n) {
                    const float d = __uint_as_float((unsigned)(w[k] >> 32));
                    dist_r[i] = d;
                    idx_r[i] = (int)(unsigned)(w[k] & 0xffffffffu);
                    if (FUSED) {
                        if (f.rearm) prow[i] = ~0ull;
                        term += (double)(f.use_sqrt ? __fsqrt_rn(d) : d);
                    }
                }
            }
        }
    } else {
        const size_t n = (size_t)B * nc;
        const size_t w0 = ((size_t)blockIdx.x * 8 + warp) * EPI_CPW;  // first column of this warp
        if (f.len_r != nullptr) {
            // ragged batch, one column at a time for the same reason: a column past its cloud's length, or of a pair whose row
            // cloud is empty, has no neighbour (and is never read); the fix-up reads the row cloud up to its length only, and the
            // loss term of a column is f(d) / (its cloud's length)
#pragma unroll 1
            for (int k = 0; k < EPI_CPW; ++k) {
                const size_t c = w0 + k;
                if (c >= n) break;  // warp-uniform
                const int b = (int)(c / nc), len = sym_len(f.len_c, b, nc);
                const int rows_b = (int)(c - (size_t)b * nc) < len ? sym_len(f.len_r, b, nr) : 0;   // warp-uniform
                const unsigned long long word = __ldcg(pcol + c);
                float d = 0.f;
                int found = -1;
                if (rows_b > 0) {
                    d = __uint_as_float((unsigned)(word >> 32));
                    found = sym_fix_column(rows + (size_t)b * nr * 3, rows_b, rows_per_block, __ldg(cols + c * 3), __ldg(cols + c * 3 + 1),
                                           __ldg(cols + c * 3 + 2), d, (int)(unsigned)(word & 0xffffffffu), lane);
                }
                if (lane == 0) {
                    dist_c[c] = d;
                    idx_c[c] = found;
                    if (FUSED) {
                        if (f.rearm) pcol[c] = ~0ull;
                        if (rows_b > 0) term += (double)(f.use_sqrt ? __fsqrt_rn(d) : d) / (double)len;
                    }
                }
            }
        } else {
            const size_t mine = w0 + (lane % EPI_CPW);
            unsigned long long my_w = 0ull;
            float mx = 0.f, my = 0.f, mz = 0.f;
            size_t my_base = 0;
            if (mine < n) {
                my_w = __ldcg(pcol + mine);
                mx = __ldg(cols + mine * 3), my = __ldg(cols + mine * 3 + 1), mz = __ldg(cols + mine * 3 + 2);
                my_base = (mine / nc) * (size_t)nr * 3;
            }
            int my_found = 0;
#pragma unroll
            for (int k = 0; k < EPI_CPW; ++k) {
                if (w0 + k >= n) break;  // warp-uniform
                const unsigned long long word = __shfl_sync(0xffffffffu, my_w, k);
                const float cx = __shfl_sync(0xffffffffu, mx, k), cy = __shfl_sync(0xffffffffu, my, k), cz = __shfl_sync(0xffffffffu, mz, k);
                const size_t base = __shfl_sync(0xffffffffu, my_base, k);
                const int found = cols_exact ? (int)(unsigned)(word & 0xffffffffu)
                                             : sym_fix_column(rows + base, nr, rows_per_block, cx, cy, cz,
                                                              __uint_as_float((unsigned)(word >> 32)), (int)(unsigned)(word & 0xffffffffu), lane);
                if (lane == k) my_found = found;
            }
            if (lane < EPI_CPW && mine < n) {
                const float d = __uint_as_float((unsigned)(my_w >> 32));
                dist_c[mine] = d;
                idx_c[mine] = my_found;
                if (FUSED) {
                    if (f.rearm) pcol[mine] = ~0ull;
                    term = (double)(f.use_sqrt ? __fsqrt_rn(d) : d);
                }
            }
        }
    }
    if (FUSED) {
        const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x, total_threads = (size_t)gridDim.x * blockDim.x;
        epi_zero_fill(f.zero[0], f.nzero[0], g, total_threads);
        epi_zero_fill(f.zero[1], f.nzero[1], g, total_threads);
        if (f.partial == nullptr) return;
        __shared__ double sh[8];
        __shared__ double sh2[2][8];
        __shared__ int is_last;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) term += __shfl_xor_sync(0xffffffffu, term, o);
        if (lane == 0) sh[warp] = term;
        __syncthreads();
        if (threadIdx.x == 0) {
            double a = 0.0;
#pragma unroll
            for (int w = 0; w < 8; ++w) a += sh[w];
            f.partial[blockIdx.x] = a;
            __threadfence();
            is_last = (atomicAdd(f.ticket, 1u) == gridDim.x - 1);
        }
        __syncthreads();
        if (!is_last) return;
        __threadfence();
        double sc = 0.0, sr = 0.0;  // fixed assignment + fixed tree => deterministic
        for (unsigned c = threadIdx.x; c < fix_blocks; c += blockDim.x) sc += __ldcg(f.partial + c);
        for (unsigned c = fix_blocks + threadIdx.x; c < gridDim.x; c += blockDim.x) sr += __ldcg(f.partial + c);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sc += __shfl_xor_sync(0xffffffffu, sc, o), sr += __shfl_xor_sync(0xffffffffu, sr, o);
        if (lane == 0) sh2[0][warp] = sc, sh2[1][warp] = sr;
        __syncthreads();
        if (threadIdx.x == 0) {
            sc = 0.0, sr = 0.0;
#pragma unroll
            for (int w = 0; w < 8; ++w) sc += sh2[0][w], sr += sh2[1][w];
            double loss = 0.0;
            if (f.fcol != 0.0) loss += f.fcol * sc;
            if (f.frow != 0.0) loss += f.frow * sr;
            // a gated scan that gave up waiting for its data (nn_sym_gated_kernel) worked on garbage: the caller sees it at
            // the first natural synchronisation point -- the loss it reads back is NaN
            if (f.err_flag != nullptr && __ldcg(f.err_flag) != 0u) loss = __longlong_as_double(0x7ff8000000000000LL);
            f.loss_out[0] = (float)loss;
            *f.ticket = 0;
        }
    }
}

}  // namespace genpc
