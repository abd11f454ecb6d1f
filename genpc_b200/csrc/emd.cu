// emd.cu -- EMD approximate matching (auction algorithm) for sm_100a: ONE persistent cooperative kernel.
//
// Replaces emd_cuda_forward (emd_cuda.cu:228-282): the reference runs `iters` x 7 launches (clear,
// calc_unass_cnt, calc_unass_cnt_sum, calc_unass_idx, Bid, GetMax, Assign) + CalcDist = 351 launches at
// iters = 50, launch-latency bound, and every Bid block re-stages the whole target cloud for <= 256 bidders.
// Here a group of CTAs owns each batch entry for the whole run:
//   * Bid, pruned form (r02, 64 <= n <= 32768): emd_sort_kernel orders the targets along a Morton curve once per call;
//     one WARP per bidder tests the bounding boxes of the 64-target blocks against the bidder's second-best bound and
//     scans only the blocks that can matter (5-7 % on the bench's inputs) -- see "pruned Bid" below;
//   * Bid, exhaustive form (other n, GENPC_EMD_PRUNE=0): an item = P unassigned points x all targets, T = 256/P threads
//     per point (P adapts so the items fill the group); targets + prices staged as float4 chunks in shared memory;
//   * the last CTA of the group to finish an iteration's bids (atomic ticket) runs the O(n) tail on its own:
//     GetMax -> Assign -> reset -> ascending compaction of the still-unassigned points, then releases a
//     per-batch flag the group spins on (iterations with 512 or more bidders spread GetMax / Assign over the
//     group between two counter barriers instead).  No grid-wide barrier, no host round trip.
// Arithmetic and tie rules are the reference's, bit for bit (oracle_emd_forward has the derivation):
//   value = (float)((3.0 - (double)sqrtf(fma(dz,dz,fma(dx,dx,dy*dy)))) - (double)price)   (emd_cuda.cu:146)
//   best / second-best with multiplicity; among equal best values the winner is the target with the smallest
//   (reference_thread(k), k) -- the order in which the reference's thread slices visit targets (:136-139,:167);
//   GetMax window +-1e-6 in double (:188); the reference's last-writer race is resolved as "highest j" (default) or
//   "lowest j" (GENPC_EMD_GETMAX=lowest): the reference itself lands on either, depending on block timing.
#include <cooperative_groups.h>
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "nn_prune.cuh"   // nn_bin_sort_kernel: counting sort over Morton cells + block boxes (same layout as emd_sort_kernel)

namespace genpc {

constexpr int EMD_THREADS = 256;
constexpr int EMD_CHUNK = 2048;  // same chunking as the reference's Bid (it defines the tie order)

struct EmdArgs {
    const float *xyz1, *xyz2;
    float *dist;
    int *assignment;
    float *price;
    int *assignment_inv, *bid;
    float *bid_increments, *max_increments;
    int *unass_idx, *unass_cnt, *max_idx;
    int *flags, *tickets, *bars;  // workspace [B] each, zeroed by the host
    float *pmin;           // workspace [B]: lowest price of the cloud at the start of the run (prices only rise)
    int B, n;
    float eps;
    int iters, group;      // group = CTAs per batch entry (1 when B >= grid)
    int two_level_div;     // two-level pre-filter while U * two_level_div >= n (0: never)
    int getmax_lowest;     // GetMax race resolved as lowest (1) or highest (0, default) bidder index
    int direct_p;          // items with at most this many bidders read the targets from global memory (no staging)
    int tail_spread_u;     // GetMax / Assign are spread over the group from this many bidders up
    // pruned Bid (r02): targets re-ordered along a Morton curve by emd_sort_kernel, (x, y, z, original index) per target,
    // and the bounding box (lo, hi) of every EMD_BLOCK consecutive sorted targets
    const float4 *tsort, *boxes;
};

struct BidState {
    float best, better;
    int bi;
};

// order in which the reference visits target k: (thread slot inside its 2048-chunk, k)
__device__ __forceinline__ long long ref_visit_key(int k, int n, int tpu_ref) {
    const int kl = k & (EMD_CHUNK - 1);
    const int end_k = min(EMD_CHUNK, n - (k - kl));
    const int delta = (end_k + tpu_ref - 1) / tpu_ref;
    return ((long long)(kl / delta) << 32) | (unsigned)k;
}

__device__ __forceinline__ void bid_merge(BidState &a, const BidState &b, int n, int tpu_ref) {
    bool take_b;
    if (b.best > a.best) take_b = true;
    else if (b.best < a.best) take_b = false;
    else if (b.bi < 0) take_b = false;
    else if (a.bi < 0) take_b = true;
    else take_b = ref_visit_key(b.bi, n, tpu_ref) < ref_visit_key(a.bi, n, tpu_ref);
    if (take_b) {
        a.better = fmaxf(b.better, a.best);
        a.best = b.best;
        a.bi = b.bi;
    } else {
        a.better = fmaxf(a.better, b.best);
    }
}

// 16-byte shared-memory load through a 32-bit shared-window address: the generic-pointer form makes ptxas rebuild the
// window base (S2UR SR_CgaCtaId + ULEA) in every iteration of the Bid scan
__device__ __forceinline__ float4 lds128(unsigned addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}

__device__ __forceinline__ int ld_acquire(const int *p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int *p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// ascending compaction of {j : assignment[j] == -1} into uidx; returns the count (valid in every thread).
// Warp w owns the contiguous slice [w * n/8, (w+1) * n/8) and walks it 128 elements at a time with one LDG.128 per lane
// (lane l holds elements 4l..4l+3 of the step: ascending order is (lane, component)).  Steps are independent, so the
// loads of a whole batch of EMD_CSTEPS steps are in flight together; the flags of the batch stay in registers between the
// counting pass and the writing pass.  One block barrier publishes the eight warp totals.  (The first form walked the
// array 256 elements at a time with two block barriers per step -- 64 barriers at n = 8192; the second one element per
// lane and step with four loads in flight -- both left the iteration's serial tail bound by L2 latency.)
constexpr int EMD_CSTEPS = 8;  // 8 x 128 = 1024 elements per warp and batch (n = 8192: the whole slice)

__device__ __noinline__ int compact_unassigned(const int *__restrict__ asg, int *__restrict__ uidx, int *__restrict__ midx, int n,
                                  int *sscan) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int WARPS = EMD_THREADS / 32;
    const int per_warp = n / WARPS;  // n % 256 == 0  =>  per_warp % 32 == 0
    const int j0 = warp * per_warp;
    const unsigned lt = (1u << lane) - 1u;
    const int4 minus1 = make_int4(-1, -1, -1, -1);
    // the LDG.128 / STG.128 forms need 16-byte aligned arrays (the C ABI takes plain pointers: fall back otherwise)
    const bool vec_ok = ((reinterpret_cast<size_t>(asg) | reinterpret_cast<size_t>(midx)) & 15) == 0;
    if (vec_ok && per_warp % 128 == 0 && per_warp <= 128 * EMD_CSTEPS) {
        // fast path (n <= 8192, n % 1024 == 0): one batch, flags kept in registers across the barrier
        const int steps = per_warp / 128;
        unsigned fl[EMD_CSTEPS];  // 4 flag bits per step
        int cnt = 0;
#pragma unroll
        for (int r = 0; r < EMD_CSTEPS; ++r) {
            fl[r] = 0;
            if (r < steps) {
                const int j = j0 + r * 128 + lane * 4;
                const int4 v = __ldcg(reinterpret_cast<const int4 *>(asg + j));
                *reinterpret_cast<int4 *>(midx + j) = minus1;  // re-arm GetMax for the next iteration
                fl[r] = (v.x == -1 ? 1u : 0u) | (v.y == -1 ? 2u : 0u) | (v.z == -1 ? 4u : 0u) | (v.w == -1 ? 8u : 0u);
            }
        }
#pragma unroll
        for (int r = 0; r < EMD_CSTEPS; ++r) cnt += __popc(fl[r]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        if (lane == 0) sscan[warp] = cnt;
        __syncthreads();
        int base = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) {
            const int c = sscan[w];
            base += (w < warp) ? c : 0;
            tot += c;
        }
#pragma unroll
        for (int r = 0; r < EMD_CSTEPS; ++r) {
            if (r < steps) {
                const unsigned b0 = __ballot_sync(0xffffffffu, fl[r] & 1u), b1 = __ballot_sync(0xffffffffu, fl[r] & 2u);
                const unsigned b2 = __ballot_sync(0xffffffffu, fl[r] & 4u), b3 = __ballot_sync(0xffffffffu, fl[r] & 8u);
                int pos = base + __popc(b0 & lt) + __popc(b1 & lt) + __popc(b2 & lt) + __popc(b3 & lt);
                const int j = j0 + r * 128 + lane * 4;
                if (fl[r] & 1u) uidx[pos++] = j;
                if (fl[r] & 2u) uidx[pos++] = j + 1;
                if (fl[r] & 4u) uidx[pos++] = j + 2;
                if (fl[r] & 8u) uidx[pos++] = j + 3;
                base += __popc(b0) + __popc(b1) + __popc(b2) + __popc(b3);
            }
        }
        __syncthreads();  // sscan may be reused
        return tot;
    }
    if (vec_ok && per_warp % (128 * EMD_CSTEPS) == 0) {
        // larger clouds (n % 8192 == 0): the same 128-element steps in batches of EMD_CSTEPS, two passes over the slice
        // (the second one re-reads it from L1 / L2 with all loads of a batch in flight again)
        int cnt = 0;
        for (int r0 = 0; r0 < per_warp; r0 += 128 * EMD_CSTEPS) {
            int4 v[EMD_CSTEPS];
#pragma unroll
            for (int r = 0; r < EMD_CSTEPS; ++r) {
                const int j = j0 + r0 + r * 128 + lane * 4;
                v[r] = __ldcg(reinterpret_cast<const int4 *>(asg + j));
                *reinterpret_cast<int4 *>(midx + j) = minus1;
            }
#pragma unroll
            for (int r = 0; r < EMD_CSTEPS; ++r) cnt += (v[r].x == -1) + (v[r].y == -1) + (v[r].z == -1) + (v[r].w == -1);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        if (lane == 0) sscan[warp] = cnt;
        __syncthreads();
        int base = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) {
            const int c = sscan[w];
            base += (w < warp) ? c : 0;
            tot += c;
        }
        if (cnt > 0) {
            for (int r0 = 0; r0 < per_warp; r0 += 128 * EMD_CSTEPS) {
                int4 v[EMD_CSTEPS];
#pragma unroll
                for (int r = 0; r < EMD_CSTEPS; ++r) v[r] = __ldcg(reinterpret_cast<const int4 *>(asg + j0 + r0 + r * 128 + lane * 4));
#pragma unroll
                for (int r = 0; r < EMD_CSTEPS; ++r) {
                    const bool f0 = v[r].x == -1, f1 = v[r].y == -1, f2 = v[r].z == -1, f3 = v[r].w == -1;
                    const unsigned b0 = __ballot_sync(0xffffffffu, f0), b1 = __ballot_sync(0xffffffffu, f1);
                    const unsigned b2 = __ballot_sync(0xffffffffu, f2), b3 = __ballot_sync(0xffffffffu, f3);
                    int pos = base + __popc(b0 & lt) + __popc(b1 & lt) + __popc(b2 & lt) + __popc(b3 & lt);
                    const int j = j0 + r0 + r * 128 + lane * 4;
                    if (f0) uidx[pos++] = j;
                    if (f1) uidx[pos++] = j + 1;
                    if (f2) uidx[pos++] = j + 2;
                    if (f3) uidx[pos++] = j + 3;
                    base += __popc(b0) + __popc(b1) + __popc(b2) + __popc(b3);
                }
            }
        }
        __syncthreads();  // sscan may be reused
        return tot;
    }
    // general path: one element per lane and step, two passes over the slice
    int cnt = 0;
#pragma unroll 8
    for (int r = 0; r < per_warp; r += 32) {
        const int j = j0 + r + lane;
        const int f = (__ldcg(asg + j) == -1);
        midx[j] = -1;
        cnt += __popc(__ballot_sync(0xffffffffu, f));
    }
    if (lane == 0) sscan[warp] = cnt;
    __syncthreads();
    int base = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) {
        const int c = sscan[w];
        base += (w < warp) ? c : 0;
        tot += c;
    }
    if (cnt > 0) {
#pragma unroll 8
        for (int r = 0; r < per_warp; r += 32) {
            const int j = j0 + r + lane;
            const int f = (__ldcg(asg + j) == -1);
            const unsigned bal = __ballot_sync(0xffffffffu, f);
            if (f) uidx[base + __popc(bal & lt)] = j;
            base += __popc(bal);
        }
    }
    __syncthreads();  // sscan may be reused
    return tot;
}

// GetMax (emd_cuda.cu:181-194: highest -- or, on request, lowest -- j inside the +-1e-6 window wins) and Assign (:196-215) for the U bidders of one
// cloud, run by ONE CTA (the iteration's serial tail).  Every bidder is a chain of dependent L2 reads
// (uidx -> bid / increment -> max_increment / max_idx -> assignment_inv, price); a thread takes EMD_TAIL_R bidders at a
// time and issues each level of the chain for all of them before it consumes any, so the tail costs about one L2
// latency per level instead of one per level and bidder.  Bidders act on disjoint targets (one winner per target), so
// the order in which they are processed does not matter.
constexpr int EMD_TAIL_R = 2;

// Both phases take the bidders u = first, first + stride, ... (first = tid, stride = EMD_THREADS when one CTA runs the tail;
// a slice per CTA when the group shares it).
__device__ __noinline__ void emd_getmax(const int *__restrict__ uidx, const int *__restrict__ bd, const float *__restrict__ binc,
                                        const float *minc, int *midx, int U, bool lowest, int first, int stride) {
    for (int u0 = first; u0 < U; u0 += stride * EMD_TAIL_R) {
        int j[EMD_TAIL_R], bid[EMD_TAIL_R];
        float inc[EMD_TAIL_R], mx[EMD_TAIL_R];
#pragma unroll
        for (int r = 0; r < EMD_TAIL_R; ++r) {
            const int u = u0 + r * stride;
            j[r] = (u < U) ? __ldcg(uidx + u) : -1;
        }
#pragma unroll
        for (int r = 0; r < EMD_TAIL_R; ++r)
            if (j[r] >= 0) bid[r] = __ldcg(bd + j[r]), inc[r] = __ldcg(binc + j[r]);
#pragma unroll
        for (int r = 0; r < EMD_TAIL_R; ++r)
            if (j[r] >= 0) mx[r] = __ldcg(minc + bid[r]);
#pragma unroll
        for (int r = 0; r < EMD_TAIL_R; ++r)
            if (j[r] >= 0 && (double)inc[r] - 1e-6 <= (double)mx[r] && (double)mx[r] <= (double)inc[r] + 1e-6)
            {
                if (lowest) atomicMin(reinterpret_cast<unsigned *>(midx + bid[r]), (unsigned)j[r]);  // -1 (re-armed) is UINT_MAX
                else atomicMax(midx + bid[r], j[r]);
            }
    }
}

__device__ __noinline__ void emd_assign(const int *__restrict__ uidx, const int *__restrict__ bd, const float *__restrict__ binc,
                                        float *minc, const int *midx, int *asg, int *asg_inv, float *pr, int U, bool last,
                                        int first, int stride) {
    for (int u0 = first; u0 < U; u0 += stride * EMD_TAIL_R) {
        int j[EMD_TAIL_R], bid[EMD_TAIL_R], win[EMD_TAIL_R], inv[EMD_TAIL_R];
        float inc[EMD_TAIL_R], p[EMD_TAIL_R];
#pragma unroll
        for (int r = 0; r < EMD_TAIL_R; ++r) {
            const int u = u0 + r * stride;
            j[r] = (u < U) ? __ldcg(uidx + u) : -1;
        }
#pragma unroll
        for (int r = 0; r < EMD_TAIL_R; ++r)
            if (j[r] >= 0) bid[r] = __ldcg(bd + j[r]), inc[r] = __ldcg(binc + j[r]);
        if (last) {
#pragma unroll
            for (int r = 0; r < EMD_TAIL_R; ++r)
                if (j[r] >= 0) {
                    asg[j[r]] = bid[r];
                    atomicMax(asg_inv + bid[r], j[r]);
                    atomicAdd(pr + bid[r], inc[r]);
                    minc[bid[r]] = -1e9f;
                }
            continue;
        }
#pragma unroll
        for (int r = 0; r < EMD_TAIL_R; ++r) win[r] = (j[r] >= 0) && (__ldcg(midx + bid[r]) == j[r]);
#pragma unroll
        for (int r = 0; r < EMD_TAIL_R; ++r)
            if (win[r]) inv[r] = __ldcg(asg_inv + bid[r]), p[r] = __ldcg(pr + bid[r]);
#pragma unroll
        for (int r = 0; r < EMD_TAIL_R; ++r)
            if (win[r]) {
                if (inv[r] != -1) asg[inv[r]] = -1;
                asg_inv[bid[r]] = j[r];
                asg[j[r]] = bid[r];
                pr[bid[r]] = __fadd_rn(p[r], inc[r]);
                minc[bid[r]] = -1e9f;
            }
    }
}

// ---- pruned Bid (r02) ------------------------------------------------------------------------------------------------
// A candidate target only matters to a bidder if its value reaches the bidder's second-best value, i.e. if
// sqrt(s) <= (3 - price) - better; every price is >= pmin0 (prices only rise), so with the targets grouped into spatially
// compact blocks a whole block is rejected by ONE test of the squared distance between the bidder and the block's bounding
// box against the same target-independent cap s_cap the two-level filter uses.  The test rejects a subset of what the
// per-target filter rejects, so the result is bit-identical to the exhaustive scan whatever the order and the grouping
// are (best / second-best with multiplicity and the (reference_thread(k), k) tie key do not depend on the visiting order).
// On the bench's inputs 5-7 % of the blocks survive in every iteration (tools/emd_prune_stats.py).
constexpr int EMD_BLOCK = 64;            // targets per block: one target PAIR per lane of the scanning warp
constexpr int EMD_PRUNE_MAX_N = 32768;   // boxes of a cloud fit the kernel's shared memory, the sort fits one CTA's
constexpr int EMD_SORT_THREADS = 1024;
// surviving blocks whose loads are in flight together.  Same-box sweep with the final structure (ms: B1 n8192 | B32 n8192 | B1
// n16384 | B20 n2048): 1: 1.32 | 2.99 | 1.65 | 1.07;  2: 1.10 | 2.50 | 1.36 | 0.89;  3: 1.10 | 2.60 | 1.41 | 0.92;
// 4: 1.17 | 2.88 | 1.47 | 0.97;  5: 1.22 | 3.12 | 1.57 | 1.01;  6: 1.36 | 3.56 | 1.67 | 1.10 (more blocks fetched before the first
// threshold exists = more targets evaluated for nothing; with the first structure, which had a separate seed block, 2 lost to 4)
#ifndef GENPC_EMD_PBATCH
#define GENPC_EMD_PBATCH 2
#endif
constexpr int EMD_PBATCH = GENPC_EMD_PBATCH;

// One CTA per cloud: Morton keys of the targets (cell << idxbits | original index), bitonic sort in shared memory, sorted
// (x, y, z, index) records and per-block bounding boxes (all lower corners, then all upper corners).  The ORDER only affects how well the blocks prune, never a result.
__global__ void __launch_bounds__(EMD_SORT_THREADS) emd_sort_kernel(const float *__restrict__ xyz2, float4 *__restrict__ tsort,
                                                                    float4 *__restrict__ boxes, int n, int np2, int idxbits,
                                                                    int mbits) {
    extern __shared__ unsigned skeys[];
    __shared__ float sred[6][EMD_SORT_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float *p2 = xyz2 + (size_t)blockIdx.x * n * 3;
    float4 *ts = tsort + (size_t)blockIdx.x * n;
    float4 *bx = boxes + (size_t)blockIdx.x * (n / EMD_BLOCK) * 2;
    const float inf = __int_as_float(0x7f800000);
    float lo[3] = {inf, inf, inf}, hi[3] = {-inf, -inf, -inf};
    for (int k = tid; k < n; k += EMD_SORT_THREADS) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float v = __ldg(p2 + k * 3 + c);
            if (fabsf(v) < inf) lo[c] = fminf(lo[c], v), hi[c] = fmaxf(hi[c], v);   // NaN / Inf do not stretch the grid
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
    __syncthreads();
    float scale[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        float l = inf, h = -inf;
        for (int w = 0; w < EMD_SORT_THREADS / 32; ++w) l = fminf(l, sred[c][w]), h = fmaxf(h, sred[3 + c][w]);
        lo[c] = l;
        const float ext = h - l;
        scale[c] = (ext > 0.f && ext < inf) ? (float)(1 << mbits) / ext : 0.f;
    }
    const int cmax = (1 << mbits) - 1;
    for (int k = tid; k < np2; k += EMD_SORT_THREADS) {
        unsigned key = 0xffffffffu;
        if (k < n) {
            unsigned code = 0;
            int cell[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float f = (__ldg(p2 + k * 3 + c) - lo[c]) * scale[c];
                cell[c] = f >= 0.f ? min((int)fminf(f, 2e9f), cmax) : 0;   // NaN -> 0
            }
            for (int bit = 0; bit < mbits; ++bit)
#pragma unroll
                for (int c = 0; c < 3; ++c) code |= (unsigned)((cell[c] >> bit) & 1) << (3 * bit + c);
            key = (code << idxbits) | (unsigned)k;
        }
        skeys[k] = key;
    }
    for (int size = 2; size <= np2; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int t = tid; t < (np2 >> 1); t += EMD_SORT_THREADS) {
                const int i = 2 * t - (t & (stride - 1));
                const unsigned u = skeys[i], v = skeys[i + stride];
                const bool up = (i & size) == 0;
                if ((u > v) == up) skeys[i] = v, skeys[i + stride] = u;
            }
        }
    }
    __syncthreads();
    const unsigned imask = (1u << idxbits) - 1u;
    for (int k = tid; k < n; k += EMD_SORT_THREADS) {
        const int o = (int)(skeys[k] & imask);
        ts[k] = make_float4(__ldg(p2 + o * 3), __ldg(p2 + o * 3 + 1), __ldg(p2 + o * 3 + 2), __int_as_float(o));
    }
    for (int blk = warp; blk < n / EMD_BLOCK; blk += EMD_SORT_THREADS / 32) {
        float l[3] = {inf, inf, inf}, h[3] = {-inf, -inf, -inf};
#pragma unroll
        for (int e = 0; e < EMD_BLOCK / 32; ++e) {
            const int o = (int)(skeys[blk * EMD_BLOCK + e * 32 + lane] & imask);
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float v = __ldg(p2 + o * 3 + c);
                l[c] = fminf(l[c], v), h[c] = fmaxf(h[c], v);   // NaN coordinates are ignored: such targets never matter
            }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                l[c] = fminf(l[c], __shfl_xor_sync(0xffffffffu, l[c], o));
                h[c] = fmaxf(h[c], __shfl_xor_sync(0xffffffffu, h[c], o));
            }
        if (lane == 0) bx[blk] = make_float4(l[0], l[1], l[2], 0.f), bx[n / EMD_BLOCK + blk] = make_float4(h[0], h[1], h[2], 0.f);
    }
}

// monotone float <-> int map (REDUX works on integers; values may be negative)
__device__ __forceinline__ int f2ord(float f) {
    const int i = __float_as_int(f);
    return i ^ ((i >> 31) & 0x7fffffff);
}
__device__ __forceinline__ float ord2f(int i) { return __int_as_float(i ^ ((i >> 31) & 0x7fffffff)); }

#ifdef GENPC_EMD_TRACE
// profiling build only (tools/emd_trace.py): phase timestamps of cloud 0, eight per iteration (0-3 phases of the
// iteration, 4-7 inside the first bidder of CTA 0 / warp 0)
__device__ unsigned long long g_emd_trace[8 * 1024];
__device__ __forceinline__ void emd_trace(int it, int k) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    if (it < 1024) g_emd_trace[it * 8 + k] = t;
}
#define EMD_TRACE(cond, it, k) do { if ((cond) && threadIdx.x == 0) emd_trace(it, k); } while (0)
#else
#define EMD_TRACE(cond, it, k) do { } while (0)
#endif

// BOXR = 0: exhaustive Bid; BOXR > 0: pruned Bid for clouds of up to BOXR * 32 blocks (box distances in BOXR registers per lane)
template <int BOXR, int MINB>
__global__ void __launch_bounds__(EMD_THREADS, MINB) emd_auction_kernel(const EmdArgs a) {
    constexpr bool PRUNE = BOXR > 0;
    // targets + prices of one chunk, two float4 planes per target PAIR p: stg[p] = (x0, x1, y0, y1), stg[EMD_CHUNK/2 + p] =
    // (z0, z1, price0, price1) -- one address register (second plane at a constant offset) and two LDS.128 per step of the
    // Bid scan (r02; four separate SoA arrays cost four LEA, four LDS.64 and six uniform address instructions per step:
    // 31 -> 21 instructions per target pair on the reject path).  Consecutive pairs are 16 B apart inside a plane, so the
    // lanes of a bidder hit distinct banks (a first r02 layout interleaved the two float4 of a pair: 32-byte lane stride,
    // 2-way conflict on every load -- 930 M of 2000 M wavefronts).
    // (PRUNE: the same array holds the cloud's block boxes instead: nblk lower corners, then nblk upper corners -- 16-byte
    // lane stride on both loads of the box test)
    __shared__ __align__(16) float4 stg[PRUNE ? 2 * BOXR * 32 : EMD_CHUNK];
    constexpr unsigned STG_PLANE = (EMD_CHUNK / 2) * 16;
    __shared__ BidState smerge[PRUNE ? 1 : EMD_THREADS];
    // PRUNE: per warp, the list of blocks that survive the box test and the queue of (original index, s) candidates
    __shared__ unsigned short s_blist[PRUNE ? EMD_THREADS / 32 : 1][PRUNE ? BOXR * 32 + EMD_PBATCH : 1];
    __shared__ float2 s_queue[PRUNE ? EMD_THREADS / 32 : 1][PRUNE ? 96 : 1];
    __shared__ int sscan[EMD_THREADS / 32];
    __shared__ int s_last;
    const int tid = threadIdx.x;
    const int n = a.n;
    const int block_cnt = n / 256;
    const unsigned stg_addr = (unsigned)__cvta_generic_to_shared(stg);

    for (int b = (a.group > 1 ? (int)blockIdx.x / a.group : (int)blockIdx.x); b < a.B;
         b += (a.group > 1 ? a.B : (int)gridDim.x)) {
        const int rank = a.group > 1 ? (int)blockIdx.x % a.group : 0;
        const float *p1 = a.xyz1 + (size_t)b * n * 3;
        const float *p2 = a.xyz2 + (size_t)b * n * 3;
        int *asg = a.assignment + (size_t)b * n;
        int *asg_inv = a.assignment_inv + (size_t)b * n;
        float *pr = a.price + (size_t)b * n;
        int *bd = a.bid + (size_t)b * n;
        float *binc = a.bid_increments + (size_t)b * n;
        float *minc = a.max_increments + (size_t)b * n;
        int *uidx = a.unass_idx + (size_t)b * n;
        int *midx = a.max_idx + (size_t)b * n;
        int *flag = a.flags + b, *ticket = a.tickets + b, *bar = a.bars + b;
        int tix_target = 0, bar_target = 0;   // arrivals expected so far (same sequence of decisions in every CTA of the group)

        if (rank == 0) {  // initial compaction (calc_unass_cnt / calc_unass_idx of iteration 0)
            const int U0 = compact_unassigned(asg, uidx, midx, n, sscan);
            // lowest initial price (0 with the reference's initial state, emd_module.py:45): the target-independent
            // pre-filter below needs a lower bound of every price, and prices only ever rise during the auction
            float pm = __int_as_float(0x7f800000);
            for (int k = tid; k < n; k += EMD_THREADS) pm = fminf(pm, __ldcg(pr + k));
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) pm = fminf(pm, __shfl_xor_sync(0xffffffffu, pm, o));
            if ((tid & 31) == 0) sscan[tid >> 5] = __float_as_int(pm);
            __threadfence();
            __syncthreads();
            if (tid == 0) {
#pragma unroll
                for (int w = 0; w < EMD_THREADS / 32; ++w) pm = fminf(pm, __int_as_float(sscan[w]));
                a.pmin[b] = pm;
                a.unass_cnt[b] = U0;
                __threadfence();
                st_release(flag, 1);
            }
        }

        if constexpr (PRUNE) {
            __syncthreads();   // the previous cloud's boxes are no longer read
            const float4 *bx = a.boxes + (size_t)b * (n / EMD_BLOCK) * 2;
            for (int k = tid; k < 2 * (n / EMD_BLOCK); k += EMD_THREADS)
                stg[k < n / EMD_BLOCK ? k : BOXR * 32 + (k - n / EMD_BLOCK)] = __ldg(bx + k);
            __syncthreads();
        }

        bool complete = false;  // every point assigned: the remaining iterations change nothing (reference: empty launches)
        for (int it = 0; it < a.iters; ++it) {
            const bool last = (it == a.iters - 1);
            if (tid == 0) {
                while (ld_acquire(flag) < it + 1) __nanosleep(64);
            }
            __syncthreads();
            const int U = __ldcg(a.unass_cnt + b);
            if (U == 0) {  // same value in every CTA of the group (read behind the same flag generation)
                complete = true;
                break;
            }
            EMD_TRACE(b == 0 && rank == 0, it, 0);   // Bid starts
            const float c_max = __fsub_rn(3.0f, __ldcg(a.pmin + b));
            const bool two_level = (a.two_level_div > 0) && ((long long)U * a.two_level_div >= n);
            // ---- Bid (emd_cuda.cu:95-179) ----
            if constexpr (PRUNE) {
                const int upb_ref = (U + block_cnt - 1) / block_cnt;
                const int tpu_ref = 256 / upb_ref;
                const int lane = tid & 31, wid = tid >> 5;
                const unsigned lt = (1u << lane) - 1u;
                const int nblk = n / EMD_BLOCK;
                const float4 *ts = a.tsort + (size_t)b * n + 2 * lane;   // lane l: sorted targets blk*64 + 2l, 2l+1
                const float inf = __int_as_float(0x7f800000);
                unsigned short *blist = s_blist[wid];
                float2 *queue = s_queue[wid];
                // One WARP per bidder.  Everything that touches L2 is issued in batches, because a bidder is otherwise a chain
                // of dependent L2 round trips (a first version that scanned the surviving blocks one after the other, each
                // with its own price gather, spent 30 us per bidder):
                //   1. box distances of all blocks (shared memory -> BOXR registers per lane)
                //   2. the EMD_PBATCH nearest blocks, loads in flight together; every lane evaluates its nearest target of the
                //      batch exactly (one price gather) -> first threshold
                //   3. the batch's other targets inside the target-independent cap s_cap are queued as (original index, s);
                //      the queue is drained 32 entries at a time (price gather, per-target filter, exact value) -> the
                //      threshold is final for most bidders
                //   4. the blocks that still pass the box test (usually 0-3) are listed and handled like 3.
                // The next bidder's index and coordinates are fetched while the current one is processed.
                const int wstride = a.group * (EMD_THREADS / 32);
                int u = rank * (EMD_THREADS / 32) + wid;
                int jn = 0;
                float xn = 0.f, yn = 0.f, zn = 0.f;
                if (u < U) {
                    jn = __ldcg(uidx + u);
                    xn = __ldg(p1 + jn * 3), yn = __ldg(p1 + jn * 3 + 1), zn = __ldg(p1 + jn * 3 + 2);
                }
                EMD_TRACE(b == 0 && rank == 0 && U > 0, it, 4);   // U, pmin known; first bidder's loads issued
                for (; u < U; u += wstride) {
                    const int j = jn;
                    const float x1 = xn, y1 = yn, z1 = zn;
#ifdef GENPC_EMD_TRACE
                    if (x1 == 123456.f) continue;   // make the timestamp below wait for the coordinates
                    EMD_TRACE(b == 0 && rank == 0 && u == 0, it, 5);
#endif
                    if (u + wstride < U) {
                        jn = __ldcg(uidx + u + wstride);
                        xn = __ldg(p1 + jn * 3), yn = __ldg(p1 + jn * 3 + 1), zn = __ldg(p1 + jn * 3 + 2);
                    }
                    BidState st;
                    st.best = -1e9f, st.better = -1e9f, st.bi = -1;
                    float bm = -2e9f;     // (lower bound of the bidder's final second-best value) - margin
                    float s_cap = inf;    // ((3 - pmin0) - bm)^2: no target beyond it can matter, whatever its price
                    auto raise_threshold = [&](float better) {
                        const float nb = __fsub_rn(better, __fmul_rn(1e-4f, fmaxf(1.f, fabsf(better))));
                        if (nb > bm) {
                            bm = nb;
                            const float tq0 = __fsub_rn(c_max, bm);
                            s_cap = tq0 > 0.f ? __fmul_rn(tq0, tq0) : -1.f;
                        }
                    };
                    auto consider = [&](int k, float s, float pk) {   // the reference's arithmetic and tie rule
                        const float d = (float)((3.0 - (double)__fsqrt_rn(s)) - (double)pk);
                        if (d > st.best) {
                            st.better = st.best;
                            st.best = d;
                            st.bi = k;
                        } else {
                            st.better = fmaxf(st.better, d);
                            if (d == st.best && ref_visit_key(k, n, tpu_ref) < ref_visit_key(st.bi, n, tpu_ref)) st.bi = k;
                        }
                        raise_threshold(st.better);
                    };
                    // per-target filter (as in the exhaustive scan) + exact evaluation
                    auto candidate = [&](int k, float s, float pk) {
                        const float tq = __fsub_rn(__fsub_rn(3.0f, pk), bm);
                        if (tq > 0.f && s <= __fmul_rn(tq, tq)) consider(k, s, pk);
                    };
                    // the warp-wide second-best value so far bounds every lane's filter: the second largest `best` of two
                    // different lanes, or the largest `better` of any lane.  Leaves bm / s_cap identical in all lanes.
                    auto share_threshold = [&]() {
                        const int ob = f2ord(st.best);
                        const int m1 = __reduce_max_sync(0xffffffffu, ob);
                        const int first = __ffs(__ballot_sync(0xffffffffu, ob == m1)) - 1;
                        const int m2 = __reduce_max_sync(0xffffffffu, lane == first ? (int)0x80000000 : ob);
                        const int mb = __reduce_max_sync(0xffffffffu, f2ord(st.better));
                        raise_threshold(ord2f(max(m2, mb)));
                    };
                    const float2 nx = make_float2(-x1, -x1), ny = make_float2(-y1, -y1), nz = make_float2(-z1, -z1);
                    // ---- 1. squared distance to every block's box, scaled DOWN by 1e-5: the reference's rounded s of a target
                    // inside the box is never below it (each difference and the fma chain are within a few 2^-24 of exact)
                    float sl[BOXR];
#pragma unroll
                    for (int r = 0; r < BOXR; ++r) {
                        const int blk = r * 32 + lane;
                        sl[r] = inf;
                        if (blk < nblk) {
                            const float4 lo = stg[blk], hi = stg[BOXR * 32 + blk];
                            const float dx = fmaxf(fmaxf(lo.x - x1, x1 - hi.x), 0.f);
                            const float dy = fmaxf(fmaxf(lo.y - y1, y1 - hi.y), 0.f);
                            const float dz = fmaxf(fmaxf(lo.z - z1, z1 - hi.z), 0.f);
                            sl[r] = __fmul_rn(__fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy))), 0.99999f);
                        }
                    }
                    // nearest remaining block as (distance bits without the low 9, block id): any near block will do; the block
                    // is removed from sl
                    auto take_nearest = [&]() {
                        unsigned key = 0xffffffffu;
#pragma unroll
                        for (int r = 0; r < BOXR; ++r) key = min(key, (__float_as_uint(sl[r]) & 0xfffffe00u) | (unsigned)(r * 32 + lane));
                        key = __reduce_min_sync(0xffffffffu, key);
                        const int blk = (int)(key & 0x1ffu);
#pragma unroll
                        for (int r = 0; r < BOXR; ++r)
                            if (r * 32 + lane == blk) sl[r] = inf;
                        return key;   // >= 0x7f800000: only +inf (taken / out of range) or NaN distances were left
                    };
                    // ---- 2. / 3. / 4. ----
                    int nq = 0;
                    auto drain = [&]() {   // the last min(nq, 32) entries of the queue
                        const int e = nq - 1 - lane;
                        if (e >= 0) {
                            const float2 qe = queue[e];
                            const int k = __float_as_int(qe.x);
                            candidate(k, qe.y, __ldcg(pr + k));
                        }
                        nq = max(nq - 32, 0);
                        __syncwarp();
                        share_threshold();
                    };
                    // the EMD_PBATCH nearest blocks open the list; the others join it once these have settled the threshold
                    int nlist = EMD_PBATCH;
#pragma unroll
                    for (int q = 0; q < EMD_PBATCH; ++q) {
                        const unsigned key = take_nearest();
                        if (lane == 0) blist[q] = (unsigned short)(key < 0x7f800000u ? (key & 0x1ffu) : nblk);
                    }
                    __syncwarp();
#pragma unroll 1
                    for (int i0 = 0; i0 < nlist; i0 += EMD_PBATCH) {
                        int bk[EMD_PBATCH];   // block ids, nblk = none; warp-uniform
                        float4 t[EMD_PBATCH][2];
#pragma unroll
                        for (int q = 0; q < EMD_PBATCH; ++q) {
                            bk[q] = i0 + q < nlist ? (int)blist[i0 + q] : nblk;
                            if (bk[q] < nblk) t[q][0] = __ldg(ts + bk[q] * EMD_BLOCK), t[q][1] = __ldg(ts + bk[q] * EMD_BLOCK + 1);
                        }
                        float2 sq[EMD_PBATCH];
#pragma unroll
                        for (int q = 0; q < EMD_PBATCH; ++q)
                            sq[q] = sqdist_ref_x2(nx, ny, nz, make_float2(t[q][0].x, t[q][1].x), make_float2(t[q][0].y, t[q][1].y),
                                                  make_float2(t[q][0].z, t[q][1].z));
                        int ev = -1;   // the target this lane has already evaluated exactly (2 * q + half)
                        if (i0 == 0) {
                            // no threshold yet: every lane evaluates its NEAREST target of the batch exactly (one price gather
                            // for the warp) -- 32 candidates that contain the bidder's nearest targets -- and the warp-wide
                            // second-best of those is the threshold for everything else
                            float smin = inf;
#pragma unroll
                            for (int q = 0; q < EMD_PBATCH; ++q) {
                                if (bk[q] < nblk) {
                                    if (sq[q].x < smin) smin = sq[q].x, ev = 2 * q;
                                    if (sq[q].y < smin) smin = sq[q].y, ev = 2 * q + 1;
                                }
                            }
                            float kw = 0.f;
#pragma unroll
                            for (int q = 0; q < EMD_PBATCH; ++q) {
                                if (ev == 2 * q) kw = t[q][0].w;
                                if (ev == 2 * q + 1) kw = t[q][1].w;
                            }
                            if (ev >= 0) {
                                const int k = __float_as_int(kw);
                                candidate(k, smin, __ldcg(pr + k));
                            }
                            share_threshold();
#ifdef GENPC_EMD_TRACE
                            if (s_cap == 123456.f) continue;
                            EMD_TRACE(b == 0 && rank == 0 && u == 0, it, 6);   // first threshold
#endif
                        }
#pragma unroll
                        for (int q = 0; q < EMD_PBATCH; ++q) {
                            if (bk[q] < nblk) {
                                const float2 s2 = sq[q];
                                const bool f0 = s2.x <= s_cap && ev != 2 * q, f1 = s2.y <= s_cap && ev != 2 * q + 1;
                                if (__any_sync(0xffffffffu, f0 || f1)) {
                                    const unsigned m0 = __ballot_sync(0xffffffffu, f0), m1 = __ballot_sync(0xffffffffu, f1);
                                    if (f0) queue[nq + __popc(m0 & lt)] = make_float2(t[q][0].w, s2.x);
                                    nq += __popc(m0);
                                    if (f1) queue[nq + __popc(m1 & lt)] = make_float2(t[q][1].w, s2.y);
                                    nq += __popc(m1);
                                    __syncwarp();
                                    while (nq >= 32) drain();   // keeps nq < 32 before the next block adds at most 64
                                }
                            }
                        }
                        if (i0 == 0) {
                            // the nearest blocks are in: settle the threshold, then list what still passes the box test
                            if (nq > 0) drain();
#pragma unroll
                            for (int r = 0; r < BOXR; ++r) {
                                const bool pass = sl[r] <= s_cap;   // taken blocks are +inf
                                const unsigned mask = __ballot_sync(0xffffffffu, pass);
                                if (pass) blist[nlist + __popc(mask & lt)] = (unsigned short)(r * 32 + lane);
                                nlist += __popc(mask);
                            }
                            __syncwarp();
                        }
                    }
                    if (nq > 0) drain();
                    // ---- merge the 32 lane states (order-independent: ties go by the reference's visit key) ----
                    {
                        const int ob = f2ord(st.best);
                        const int m1 = __reduce_max_sync(0xffffffffu, ob);
                        const unsigned tie = __ballot_sync(0xffffffffu, ob == m1);
                        if (__popc(tie) == 1) {
                            // one lane holds the best value: second-best = the larger of the other lanes' best and anybody's better
                            const int src = __ffs(tie) - 1;
                            const int m2 = __reduce_max_sync(0xffffffffu, lane == src ? (int)0x80000000 : ob);
                            const int mb = __reduce_max_sync(0xffffffffu, f2ord(st.better));
                            st.bi = __shfl_sync(0xffffffffu, st.bi, src);
                            st.best = ord2f(m1);
                            st.better = ord2f(max(m2, mb));
                        } else {
#pragma unroll 1
                            for (int o = 16; o > 0; o >>= 1) {
                                BidState ot;
                                ot.best = __shfl_down_sync(0xffffffffu, st.best, o);
                                ot.better = __shfl_down_sync(0xffffffffu, st.better, o);
                                ot.bi = __shfl_down_sync(0xffffffffu, st.bi, o);
                                bid_merge(st, ot, n, tpu_ref);
                            }
                        }
                    }
                    if (lane == 0) {
                        const float inc = __fadd_rn(__fsub_rn(st.best, st.better), a.eps);
                        bd[j] = st.bi;
                        binc[j] = inc;
                        atomicMax(reinterpret_cast<int *>(minc + st.bi), __float_as_int(inc));  // inc > 0
                    }
                    __syncwarp();   // the next bidder reuses the warp's list and queue
                    EMD_TRACE(b == 0 && rank == 0 && u == 0, it, 7);   // first bidder done
                }
            } else if (U > 0) {
                const int upb_ref = (U + block_cnt - 1) / block_cnt;
                const int tpu_ref = 256 / upb_ref;
                // points per item: spread the U bidders over the group; every item re-stages the whole target cloud, so
                // fewer, fuller items win (a rounds*P balance model measured 3x slower at B=32: staging dominated)
                int P = (U + a.group - 1) / a.group;
                P = max(1, min(P, EMD_THREADS));
                const int T = EMD_THREADS / P;
                const int items = (U + P - 1) / P;
                for (int g = rank; g < items; g += a.group) {
                    const int ps = tid / T, tpt = tid - ps * T;
                    const int u = g * P + ps;
                    const bool active = (ps < P) && (u < U);
                    int j = -1;
                    float x1 = 0.f, y1 = 0.f, z1 = 0.f;
                    if (active) {
                        j = __ldcg(uidx + u);
                        x1 = __ldg(p1 + j * 3), y1 = __ldg(p1 + j * 3 + 1), z1 = __ldg(p1 + j * 3 + 2);
                    }
                    BidState st;
                    st.best = -1e9f, st.better = -1e9f, st.bi = -1;
                    float bm = -2e9f;   // better - margin (pre-filter threshold)
                    float s_cap = __int_as_float(0x7f800000);  // target-independent bound on s (two-level filter)
                    // exact evaluation of one candidate (the reference's arithmetic and tie rule)
                    auto consider = [&](int k, float s, float pk) {
                        const float d = (float)((3.0 - (double)__fsqrt_rn(s)) - (double)pk);
                        if (d > st.best) {
                            st.better = st.best;
                            st.best = d;
                            st.bi = k;
                        } else {
                            st.better = fmaxf(st.better, d);
                            if (d == st.best && ref_visit_key(k, n, tpu_ref) < ref_visit_key(st.bi, n, tpu_ref)) st.bi = k;
                        }
                        bm = __fsub_rn(st.better, __fmul_rn(1e-4f, fmaxf(1.f, fabsf(st.better))));
                        // every price >= pmin0, so a candidate that matters has sqrt(s) <= (3 - pmin0) - bm, whatever its target
                        const float tq0 = __fsub_rn(c_max, bm);
                        s_cap = tq0 > 0.f ? __fmul_rn(tq0, tq0) : -1.f;
                    };
                    // two targets per step on the packed FP32 pipe.  Conservative pre-filter (no sqrt, no FP64): a
                    // candidate can only matter if its value d >= better, i.e. sqrt(s) <= 3 - price - better up to a few
                    // ulps; bm = better - margin with margin = 1e-4*max(1,|better|) (hundreds of ulps) makes
                    // "tq > 0 && s <= tq^2" a superset of those candidates; whatever passes takes the exact path above,
                    // so the result is bit-identical to evaluating every candidate exactly.
                    const float2 nx = make_float2(-x1, -x1), ny = make_float2(-y1, -y1), nz = make_float2(-z1, -z1);
                    auto step2 = [&](int k, float2 tx, float2 ty, float2 tz, float2 pk) {
                        const float2 tc = make_float2(__fsub_rn(3.0f, pk.x), __fsub_rn(3.0f, pk.y));
                        const float2 s2 = sqdist_ref_x2(nx, ny, nz, tx, ty, tz);
                        const float2 tq = __fadd2_rn(tc, make_float2(-bm, -bm));
                        const float2 tq2 = __fmul2_rn(tq, tq);
                        const bool c0 = tq.x > 0.f && s2.x <= tq2.x;
                        const bool c1 = tq.y > 0.f && s2.y <= tq2.y;
                        if (c0) consider(k, s2.x, pk.x);
                        // bm may have risen while handling the first candidate; the filter stays conservative because it
                        // was evaluated against the OLDER (lower) threshold
                        if (c1) consider(k + 1, s2.y, pk.y);
                    };
                    if (P <= a.direct_p) {
                        // thin items (few bidders per CTA, the late iterations): staging the whole target cloud through
                        // shared memory for a handful of points costs more than the scan itself -- read the targets
                        // straight from global memory (L1/L2 resident: 16 B per target), no block barriers
                        if (active) {
                            const float2 *t2 = reinterpret_cast<const float2 *>(p2);   // 3 float2 per target pair
                            const float2 *pr2 = reinterpret_cast<const float2 *>(pr);
#pragma unroll 2
                            for (int kp = tpt; kp < (n >> 1); kp += T) {                // n is even (n % 256 == 0)
                                const float2 q0 = __ldg(t2 + kp * 3), q1 = __ldg(t2 + kp * 3 + 1), q2 = __ldg(t2 + kp * 3 + 2);
                                const float2 pk = __ldcg(pr2 + kp);
                                // q0 = (x0, y0), q1 = (z0, x1), q2 = (y1, z1)
                                step2(2 * kp, make_float2(q0.x, q1.y), make_float2(q0.y, q2.x), make_float2(q1.x, q2.y), pk);
                            }
                        }
                    } else
                    for (int k2 = 0; k2 < n; k2 += EMD_CHUNK) {
                        const int end_k = min(EMD_CHUNK, n - k2);
                        __syncthreads();
                        for (int k = tid; k < end_k; k += EMD_THREADS) {
                            const float *tp = p2 + (size_t)(k2 + k) * 3;
                            float *q = reinterpret_cast<float *>(stg + (k >> 1)) + (k & 1);
                            q[0] = __ldg(tp), q[2] = __ldg(tp + 1);
                            q[STG_PLANE / 4] = __ldg(tp + 2), q[STG_PLANE / 4 + 2] = __ldcg(pr + k2 + k);
                        }
                        __syncthreads();
                        if (active && two_level) {
                            // early iterations (most points still bid, prices near their start): one compare per target
                            // against the target-independent bound s_cap rejects almost everything before the price is
                            // even read; survivors take the per-target filter + exact path.  Half the instructions of the
                            // single-level loop while prices are small; later (bound loose) the single-level loop is used.
                            unsigned sa = stg_addr + (unsigned)tpt * 16u;
                            for (int kp = tpt; kp < (end_k >> 1); kp += T, sa += (unsigned)T * 16u) {
                                const float4 q0 = lds128(sa), q1 = lds128(sa + STG_PLANE);
                                const float2 s2 = sqdist_ref_x2(nx, ny, nz, make_float2(q0.x, q0.y), make_float2(q0.z, q0.w),
                                                                make_float2(q1.x, q1.y));
                                if (s2.x <= s_cap || s2.y <= s_cap) {
                                    const float2 pk = make_float2(q1.z, q1.w);
                                    const float tq_x = __fsub_rn(__fsub_rn(3.0f, pk.x), bm);
                                    if (tq_x > 0.f && s2.x <= __fmul_rn(tq_x, tq_x)) consider(k2 + 2 * kp, s2.x, pk.x);
                                    const float tq_y = __fsub_rn(__fsub_rn(3.0f, pk.y), bm);   // bm as updated by the first
                                    if (tq_y > 0.f && s2.y <= __fmul_rn(tq_y, tq_y)) consider(k2 + 2 * kp + 1, s2.y, pk.y);
                                }
                            }
                        } else if (active) {
                            unsigned sa = stg_addr + (unsigned)tpt * 16u;
#pragma unroll 2
                            for (int kp = tpt; kp < (end_k >> 1); kp += T, sa += (unsigned)T * 16u) {   // end_k is even (n % 256 == 0)
                                const float4 q0 = lds128(sa), q1 = lds128(sa + STG_PLANE);
                                step2(k2 + 2 * kp, make_float2(q0.x, q0.y), make_float2(q0.z, q0.w), make_float2(q1.x, q1.y),
                                      make_float2(q1.z, q1.w));
                            }
                        }
                    }
                    // merge the T partial states of each point (tree over shared memory)
                    __syncthreads();
                    smerge[tid] = st;
                    __syncthreads();
                    for (int stride = 1; stride < T; stride <<= 1) {
                        if (active && (tpt % (2 * stride)) == 0 && tpt + stride < T) {
                            BidState mine = smerge[tid];
                            bid_merge(mine, smerge[tid + stride], n, tpu_ref);
                            smerge[tid] = mine;
                        }
                        __syncthreads();
                    }
                    if (active && tpt == 0) {
                        const BidState r = smerge[tid];
                        const float inc = __fadd_rn(__fsub_rn(r.best, r.better), a.eps);
                        bd[j] = r.bi;
                        binc[j] = inc;
                        atomicMax(reinterpret_cast<int *>(minc + r.bi), __float_as_int(inc));  // inc > 0
                    }
                }
            }
            // ---- tail of the iteration: GetMax -> Assign -> compaction ----
            // Few bidders (the common case): the last CTA that bid (atomic ticket; CTAs without a bidder do not take part in
            // the pruned form) runs all three on its own -- no group-wide barrier.  Many bidders (the first iterations; one
            // CTA would spend up to 90 us on them at n = 16384): GetMax and Assign are spread over the group between two
            // counter barriers, the last CTA to finish Assign compacts.
            const int work_ctas = (PRUNE && a.group > 1) ? min(a.group, (U + EMD_THREADS / 32 - 1) / (EMD_THREADS / 32)) : a.group;
            const bool spread = a.group > 1 && U >= a.tail_spread_u;
            auto group_barrier = [&]() {
                __threadfence();
                __syncthreads();
                bar_target += a.group;
                if (tid == 0) {
                    atomicAdd(bar, 1);
                    while (ld_acquire(bar) < bar_target) {
                    }
                }
                __syncthreads();
            };
            if (spread) {
                group_barrier();   // every bid of the cloud is in
                emd_getmax(uidx, bd, binc, minc, midx, U, a.getmax_lowest != 0, rank * EMD_THREADS + tid, a.group * EMD_THREADS);
                group_barrier();
                emd_assign(uidx, bd, binc, minc, midx, asg, asg_inv, pr, U, last, rank * EMD_THREADS + tid, a.group * EMD_THREADS);
            }
            const bool takes_ticket = spread || rank < work_ctas;
            const int arrivals = spread ? a.group : work_ctas;
            if (takes_ticket) {
                __threadfence();
                __syncthreads();
                if (tid == 0) s_last = (a.group == 1) || (atomicAdd(ticket, 1) == tix_target + arrivals - 1);
                __syncthreads();
            }
            tix_target += arrivals;
            if (takes_ticket && s_last) {
                EMD_TRACE(b == 0, it, 1);   // every CTA of the group has bid
                __threadfence();
                if (!spread) {
                    emd_getmax(uidx, bd, binc, minc, midx, U, a.getmax_lowest != 0, tid, EMD_THREADS);
                    __syncthreads();
                    emd_assign(uidx, bd, binc, minc, midx, asg, asg_inv, pr, U, last, tid, EMD_THREADS);
                    __syncthreads();
                }
                EMD_TRACE(b == 0, it, 2);
                const int U2 = compact_unassigned(asg, uidx, midx, n, sscan);
                __threadfence();
                __syncthreads();
                if (tid == 0) {
                    a.unass_cnt[b] = U2;
                    __threadfence();
                    st_release(flag, it + 2);
                }
                EMD_TRACE(b == 0, it, 3);   // released
            }
        }
        // ---- CalcDist (:217-226), split over the group ----
        if (tid == 0 && !complete) {
            while (ld_acquire(flag) < a.iters + 1) __nanosleep(64);
        }
        __syncthreads();
        for (int j = rank * EMD_THREADS + tid; j < n; j += a.group * EMD_THREADS) {
            const int k = __ldcg(asg + j);
            const float dx = __fsub_rn(__ldg(p1 + j * 3), __ldg(p2 + k * 3));
            const float dy = __fsub_rn(__ldg(p1 + j * 3 + 1), __ldg(p2 + k * 3 + 1));
            const float dz = __fsub_rn(__ldg(p1 + j * 3 + 2), __ldg(p2 + k * 3 + 2));
            a.dist[(size_t)b * n + j] = __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
        }
        __syncthreads();
    }
}

// NmDistanceGradKernel of emd_cuda.cu:284-300: gradient to xyz1 only, ACCUMULATED (atomicAdd in the reference,
// one term per element so a plain read-add-write is identical).
__global__ void emd_grad_kernel(const float *__restrict__ xyz1, const float *__restrict__ xyz2,
                                const float *__restrict__ graddist, const int *__restrict__ idx, float *gradxyz, int B,
                                int n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)B * n) return;
    const size_t b = i / n;
    const size_t t = b * n + __ldg(idx + i);
    const float g = __fmul_rn(__ldg(graddist + i), 2.f);
#pragma unroll
    for (int c = 0; c < 3; ++c)
        gradxyz[i * 3 + c] = __fadd_rn(gradxyz[i * 3 + c], __fmul_rn(g, __fsub_rn(__ldg(xyz1 + i * 3 + c), __ldg(xyz2 + t * 3 + c))));
}

}  // namespace genpc

using namespace genpc;

#ifdef GENPC_EMD_TRACE
extern "C" int genpc_emd_trace_read(unsigned long long *host, int count) {
    return (int)cudaMemcpyFromSymbol(host, g_emd_trace, sizeof(unsigned long long) * count);
}
#endif

// The forward's workspace: the control words (flags, tickets, lowest prices, barriers: B each, then four scratch words of the
// sort's range check) and, for the pruned Bid, from the next 256-byte offset the sorted targets and their block boxes
struct EmdWs {
    size_t bytes;
    int *ctl;
    float4 *tsort, *boxes;
};
static EmdWs emd_layout(int B, int n, bool pruned, void *base = nullptr) {
    WsCursor c{static_cast<char *>(base)};
    EmdWs w = {};
    w.ctl = c.take<int>(4 * (size_t)B + 4);
    if (pruned) w.tsort = c.take<float4>((size_t)B * n, 256), w.boxes = c.take<float4>((size_t)B * (n / EMD_BLOCK) * 2);
    return w.bytes = c.bytes(), w;
}

extern "C" size_t genpc_emd_workspace_bytes(int B) { return B < 0 ? 0 : emd_layout(B, 0, false).bytes; }

static bool emd_prune_feasible(int n) { return n >= EMD_BLOCK && n % EMD_BLOCK == 0 && n <= EMD_PRUNE_MAX_N; }

extern "C" size_t genpc_emd_workspace_bytes_n(int B, int n) { return B < 0 || n < 0 ? 0 : emd_layout(B, n, emd_prune_feasible(n)).bytes; }

extern "C" int genpc_emd_forward(const float *xyz1, const float *xyz2, float *dist, int *assignment, float *price,
                                 int *assignment_inv, int *bid, float *bid_increments, float *max_increments,
                                 int *unass_idx, int *unass_cnt, int *max_idx, int B, int n, int m, float eps, int iters,
                                 void *workspace, size_t workspace_bytes, genpc_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    // the reference's checks (emd_cuda.cu:236-249)
    if (n != m || B > 512 || n % 256 != 0 || B < 0 || n < 0) return GENPC_ERR_SHAPE;
    // eps <= 0: the bid increments best - better + eps are no longer all positive and the integer atomicMax over their bit
    // patterns would order them differently from the reference's float atomicMax; iters <= 0 leaves assignment = -1 and the
    // distance / gradient kernels would index xyz2[-1] (the reference does, emd_cuda.cu:217-226).  Both rejected (ADVICE r01).
    if (!(eps > 0.f) || iters <= 0) return GENPC_ERR_SHAPE;
    if (B == 0 || n == 0) return GENPC_OK;
    if (workspace == nullptr || workspace_bytes < genpc_emd_workspace_bytes(B)) return GENPC_ERR_WORKSPACE;
    cudaError_t e = cudaMemsetAsync(workspace, 0, genpc_emd_workspace_bytes(B), stream);
    if (e != cudaSuccess) return (int)e;
    // pruned Bid: default whenever the caller's workspace holds the sorted copy (genpc_emd_workspace_bytes_n) and the cloud is
    // large enough for the sort to pay; GENPC_EMD_PRUNE=0 forces the exhaustive scan, =1 the pruned one wherever feasible
    const char *pt = tunable("GENPC_EMD_PRUNE");
    const int prune_knob = pt != nullptr ? atoi(pt) : -1;
    bool prune = emd_prune_feasible(n) && workspace_bytes >= genpc_emd_workspace_bytes_n(B, n) &&
                 (reinterpret_cast<size_t>(workspace) & 15) == 0;
    // measured (ms, exhaustive / pruned): 1 x 1024: 0.63 / 0.71, 32 x 1024: 1.06 / 0.88, 1 x 2048: 0.77 / 0.75, 8 x 4096: 2.00 / 1.01,
    // 2 x 32768: 10.6 / 2.44
    if (prune_knob == 0 || (prune_knob < 0 && (n < 1024 || (n < 2048 && (long long)B * n < 16384)))) prune = false;
    int dev = 0, sms = 0, per_sm = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // pruned: three CTAs per SM (80 registers) beat four (64 registers, spills) on every shape of a same-box A/B
    // (profiles/r02k_emd_prune.txt)
    void *kernel = (void *)emd_auction_kernel<0, 5>;
    if (prune) {
        const int nblk = n / EMD_BLOCK;
        if (nblk <= 128) kernel = (void *)emd_auction_kernel<4, 3>;
        else if (nblk <= 256) kernel = (void *)emd_auction_kernel<8, 3>;
        else kernel = (void *)emd_auction_kernel<16, 3>;
    }
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, EMD_THREADS, 0);
    if (e != cudaSuccess) return (int)e;
    const int resident = sms * per_sm;
    if (resident <= 0) return (int)cudaErrorLaunchOutOfResources;
    const EmdWs w = emd_layout(B, n, prune, workspace);
    EmdArgs a = {};
    a.xyz1 = xyz1, a.xyz2 = xyz2, a.dist = dist, a.assignment = assignment, a.price = price;
    a.assignment_inv = assignment_inv, a.bid = bid, a.bid_increments = bid_increments;
    a.max_increments = max_increments, a.unass_idx = unass_idx, a.unass_cnt = unass_cnt, a.max_idx = max_idx;
    a.flags = w.ctl, a.tickets = w.ctl + B, a.pmin = (float *)(w.ctl + 2 * (size_t)B), a.bars = w.ctl + 3 * (size_t)B;
    a.B = B, a.n = n, a.eps = eps, a.iters = iters;
    int grid;
    if (B >= resident) {
        a.group = 1;
        grid = resident;
    } else {
        a.group = resident / B;
        // more CTAs than 256-point items in the first (all-unassigned) iteration is wasted spinning
        const int useful = (n + 15) / 16;
        if (a.group > useful) a.group = useful;
        if (a.group < 1) a.group = 1;
        grid = a.group * B;
    }
    // measured on B200 (profiles/r01j_emd_direct.txt)
    a.direct_p = 8;
    // same-box sweep (ms: B1 n8192 | B32 n8192 | B1 n16384 | B20 n2048): 64: 1.10 | 2.48 | 1.24 | 0.99;  256: 1.08 | 2.47 | 1.24 | 0.91;
    // 512: 1.04 | 2.45 | 1.23 | 0.90;  1024: 1.08 | 2.48 | 1.31 | 0.90;  2048: 1.10 | 2.51 | 1.38 | 0.89;  4096: 1.12 | 2.53 | 1.43 | 0.90
    a.tail_spread_u = 512;
    a.two_level_div = 8;
    const char *gm = tunable("GENPC_EMD_GETMAX");  // "lowest": the other legitimate outcome of the reference's race
    a.getmax_lowest = (gm != nullptr && strcmp(gm, "lowest") == 0) ? 1 : 0;
    if ((reinterpret_cast<size_t>(xyz2) & 7) != 0 || (reinterpret_cast<size_t>(price) & 7) != 0) a.direct_p = 0;  // LDG.64
    if (prune) {
        int np2 = 1, idxbits = 0;
        while (np2 < n) np2 <<= 1, ++idxbits;
        int mbits = (31 - idxbits) / 3;   // cell << idxbits | index stays below the 0xffffffff padding key
        if (mbits > 10) mbits = 10;
        const size_t smem = (size_t)np2 * sizeof(unsigned);
        static bool attr_set[64] = {};
        if (smem > 48 * 1024 && !(dev < 64 && attr_set[dev])) {
            e = cudaFuncSetAttribute(emd_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024);
            if (e != cudaSuccess) return (int)e;
            if (dev < 64) attr_set[dev] = true;
        }
        // default: counting sort over grid cells (nn_bin_sort_kernel; the order inside a cell is whatever the shared-memory
        // atomics give, which shapes the blocks but never a result) -- 40-100 us faster per call than the bitonic sort of
        // (Morton key, index) words, which GENPC_EMD_SORT=bitonic still selects (deterministic block contents)
        const char *sk = tunable("GENPC_EMD_SORT");
        if (sk == nullptr || strcmp(sk, "bitonic") != 0) {
            PruneSortParams sp = {};
            sp.xyz[0] = xyz2, sp.xyz[1] = xyz2, sp.n[0] = n, sp.n[1] = n, sp.B = B, sp.limit = 3.0e38f;
            sp.sorted[0] = sp.sorted[1] = w.tsort, sp.boxes[0] = sp.boxes[1] = w.boxes;
            sp.ctl = w.ctl + 4 * (size_t)B;   // scratch words of the range check (unused here)
            sp.hilbert = (sk == nullptr || strcmp(sk, "morton") != 0) ? 1 : 0;
            nn_bin_sort_kernel<1><<<B, PR_SORT_THREADS, 0, stream>>>(sp);   // grid = B: side 0 only
        } else {
            emd_sort_kernel<<<B, EMD_SORT_THREADS, smem, stream>>>(xyz2, w.tsort, w.boxes, n, np2, idxbits, mbits);
        }
        GENPC_CHECK_LAUNCH();
        a.tsort = w.tsort, a.boxes = w.boxes;
    }
    void *kargs[] = {(void *)&a};
    e = cudaLaunchCooperativeKernel(kernel, dim3(grid), dim3(EMD_THREADS), kargs, 0, stream);
    if (e != cudaSuccess) return (int)e;
    return GENPC_OK;
}

extern "C" int genpc_emd_backward(const float *xyz1, const float *xyz2, float *gradxyz, const float *graddist,
                                  const int *idx, int B, int n, genpc_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (B < 0 || n < 0) return GENPC_ERR_SHAPE;
    const size_t tot = (size_t)B * n;
    if (tot == 0) return GENPC_OK;
    emd_grad_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, stream>>>(xyz1, xyz2, graddist, idx, gradxyz, B, n);
    GENPC_CHECK_LAUNCH();
    return GENPC_OK;
}
