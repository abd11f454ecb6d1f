// knn.cu -- mean distance to the k nearest neighbours of every point of a cloud, or of each cloud of a batch (k <= 32),
// for sm_100a.
//
// The fusion tail of reg() ends with Open3D's remove_statistical_outlier(nb_neighbors=20, std_ratio) on the fused cloud
// (reg_xyz.py:219, utils/dataUtils.py:652-666; third-party CPU KD-tree code, not vendored): per point the mean distance
// to its nb_neighbors nearest neighbours, then a mean + std_ratio * std threshold over the cloud.  The per-point part is a
// k-NN extension of the Chamfer scan (SURVEY.md section 8f.3):
//   * four adjacent lanes per query point (each scans a quarter of every tile; the four sorted lists are merged by a
//     shuffle butterfly at the end), the cloud swept through shared memory in SoA tiles (LDS.128);
//   * squared distance with the Chamfer rounding order fma(dz,dz,fma(dx,dx,dy*dy));
//   * the k smallest squared distances are kept SORTED in registers; a candidate below the current k-th value is
//     inserted by a branch-free min/max ripple (2 instructions per slot), others cost one compare;
//   * mean = (sum of sqrt of the k values, added in ascending order in fp32) / k  -- order fixed => bit-reproducible,
//     mirrored by oracle_knn_mean_distance.
// include_self != 0 counts the point itself (distance 0) among the k, as Open3D's KD-tree query of a cloud point does.
// A batch of clouds is one launch: cloud b is blockIdx.y, its first len[b] rows of a common stride are its points.  A cloud's
// CTAs, tiles and lane clamps are those of a solo call on its points alone, so every cloud gets the solo call's bits.
#include "common.cuh"

namespace genpc {

constexpr int KNN_THREADS = 128;
constexpr int KNN_SPLIT = 4;    // lanes per query point: each scans a quarter of every tile, lists merged by shuffles
constexpr int KNN_TILE = 2048;  // targets staged per step (24 KB)

// insert v into the ascending list best[0..K) (branch-free ripple, 2 instructions per slot)
template <int K>
__device__ __forceinline__ void knn_insert(float (&best)[K], float v) {
#pragma unroll
    for (int c = 0; c < K; ++c) {
        const float lo = fminf(best[c], v);
        v = fmaxf(best[c], v);
        best[c] = lo;
    }
}

// xyz [B][stride][3], mean_out [B][stride]; len [B] (NULL: every cloud fills the stride) is clamped to [0, stride] here.
// Rows past a cloud's length are never read and get -1 (Open3D's "the query found nothing").
template <int K>
__global__ void __launch_bounds__(KNN_THREADS) knn_mean_kernel(const float *__restrict__ xyz, int stride,
                                                               const int *__restrict__ len, int include_self,
                                                               float *__restrict__ mean_out) {
    __shared__ __align__(16) float s[3][KNN_TILE];
    xyz += (size_t)blockIdx.y * stride * 3;
    mean_out += (size_t)blockIdx.y * stride;
    const int n = len ? min(max(__ldg(len + blockIdx.y), 0), stride) : stride;
    // KNN_SPLIT adjacent lanes share one query (a thread per query leaves one warp per scheduler on a 20 000-point cloud:
    // latency bound); out-of-range queries are clamped so that whole lane groups stay converged for the shuffles
    const int q0 = blockIdx.x * (KNN_THREADS / KNN_SPLIT);
    if (q0 >= n) {  // the whole CTA lies in the padding: its rows get -1 and it leaves before the first barrier
        if (threadIdx.x < KNN_THREADS / KNN_SPLIT && q0 + threadIdx.x < stride) mean_out[q0 + threadIdx.x] = -1.0f;
        return;
    }
    const int q = (blockIdx.x * KNN_THREADS + threadIdx.x) / KNN_SPLIT, sub = threadIdx.x & (KNN_SPLIT - 1);
    const bool valid = q < n;
    const int i = valid ? q : n - 1;
    const float qx = __ldg(xyz + (size_t)i * 3), qy = __ldg(xyz + (size_t)i * 3 + 1), qz = __ldg(xyz + (size_t)i * 3 + 2);
    const float inf = __int_as_float(0x7f800000);
    float best[K];
#pragma unroll
    for (int c = 0; c < K; ++c) best[c] = inf;
    const float4 *sx4 = reinterpret_cast<const float4 *>(s[0]);
    const float4 *sy4 = reinterpret_cast<const float4 *>(s[1]);
    const float4 *sz4 = reinterpret_cast<const float4 *>(s[2]);
    for (int t0 = 0; t0 < n; t0 += KNN_TILE) {
        const int cnt = min(KNN_TILE, n - t0);
        const int cnt4 = (cnt + 3) & ~3;
        __syncthreads();
        for (int k = threadIdx.x; k < cnt4; k += KNN_THREADS) {
            float x = inf, y = inf, z = inf;  // padding: distance = +inf, never inserted
            if (k < cnt) x = __ldg(xyz + (size_t)(t0 + k) * 3), y = __ldg(xyz + (size_t)(t0 + k) * 3 + 1), z = __ldg(xyz + (size_t)(t0 + k) * 3 + 2);
            s[0][k] = x, s[1][k] = y, s[2][k] = z;
        }
        __syncthreads();
        for (int g = sub; g < cnt4 / 4; g += KNN_SPLIT) {
            const float4 X = sx4[g], Y = sy4[g], Z = sz4[g];
            float d[4];
            d[0] = sqdist_ref(qx, qy, qz, X.x, Y.x, Z.x);
            d[1] = sqdist_ref(qx, qy, qz, X.y, Y.y, Z.y);
            d[2] = sqdist_ref(qx, qy, qz, X.z, Y.z, Z.z);
            d[3] = sqdist_ref(qx, qy, qz, X.w, Y.w, Z.w);
            if (!include_self) {
                const int self = i - (t0 + g * 4);
                if (self >= 0 && self < 4) d[self] = inf;
            }
            if (fmin3(fminf(d[0], d[1]), d[2], d[3]) < best[K - 1]) {  // rare once the list has settled
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if (d[e] < best[K - 1]) knn_insert<K>(best, d[e]);
            }
        }
    }
    // merge the KNN_SPLIT lists of a query: butterfly over the lane group, every lane ends with the same K smallest values
#pragma unroll
    for (int o = 1; o < KNN_SPLIT; o <<= 1) {
        float other[K];
#pragma unroll
        for (int c = 0; c < K; ++c) other[c] = __shfl_xor_sync(0xffffffffu, best[c], o);
#pragma unroll
        for (int c = 0; c < K; ++c)
            if (other[c] < best[K - 1]) knn_insert<K>(best, other[c]);
    }
    if (sub != 0 || q >= stride) return;
    if (!valid) {
        mean_out[q] = -1.0f;
        return;
    }
    float sum = 0.f;
    int m = 0;
#pragma unroll
    for (int c = 0; c < K; ++c) {
        if (best[c] < inf) {
            sum = __fadd_rn(sum, __fsqrt_rn(best[c]));
            ++m;
        }
    }
    mean_out[q] = m > 0 ? __fdiv_rn(sum, (float)m) : -1.0f;  // Open3D: mean = -1 when the query finds nothing
}

}  // namespace genpc

using namespace genpc;

// One cloud per grid row; genpc_knn_mean_distance is the B = 1, len = NULL case (a 1-D grid).
static int knn_launch(const float *xyz, const int *len, int B, int n, int k, int include_self, float *mean_dist,
                      cudaStream_t stream) {
    if (n == 0) return GENPC_OK;
    const dim3 grid((unsigned)(((size_t)n * KNN_SPLIT + KNN_THREADS - 1) / KNN_THREADS), (unsigned)B);
#define KNN_CASE(KK) \
    if (k <= KK) { knn_mean_kernel<KK><<<grid, KNN_THREADS, 0, stream>>>(xyz, n, len, include_self, mean_dist); GENPC_CHECK_LAUNCH(); return GENPC_OK; }
    // a list longer than k is NOT equivalent (the mean runs over the whole list), so every k has its own size
    switch (k) {
        case 1: KNN_CASE(1) case 2: KNN_CASE(2) case 3: KNN_CASE(3) case 4: KNN_CASE(4) case 5: KNN_CASE(5)
        case 6: KNN_CASE(6) case 7: KNN_CASE(7) case 8: KNN_CASE(8) case 9: KNN_CASE(9) case 10: KNN_CASE(10)
        case 11: KNN_CASE(11) case 12: KNN_CASE(12) case 13: KNN_CASE(13) case 14: KNN_CASE(14) case 15: KNN_CASE(15)
        case 16: KNN_CASE(16) case 17: KNN_CASE(17) case 18: KNN_CASE(18) case 19: KNN_CASE(19) case 20: KNN_CASE(20)
        case 21: KNN_CASE(21) case 22: KNN_CASE(22) case 23: KNN_CASE(23) case 24: KNN_CASE(24) case 25: KNN_CASE(25)
        case 26: KNN_CASE(26) case 27: KNN_CASE(27) case 28: KNN_CASE(28) case 29: KNN_CASE(29) case 30: KNN_CASE(30)
        case 31: KNN_CASE(31) default: KNN_CASE(32)
    }
#undef KNN_CASE
    return GENPC_ERR_SHAPE;
}

extern "C" int genpc_knn_mean_distance(const float *xyz, int n, int k, int include_self, float *mean_dist,
                                       genpc_stream_t stream) {
    if (n < 0 || k < 1 || k > 32) return GENPC_ERR_SHAPE;
    return knn_launch(xyz, nullptr, 1, n, k, include_self, mean_dist, (cudaStream_t)stream);
}

extern "C" int genpc_knn_mean_distance_ragged(const float *xyz, const int *len, int B, int n, int k, int include_self,
                                              float *mean_dist, genpc_stream_t stream) {
    if (!xyz || !len || !mean_dist || B < 1 || B > 65535 || n < 0 || k < 1 || k > 32) return GENPC_ERR_SHAPE;
    return knn_launch(xyz, len, B, n, k, include_self, mean_dist, (cudaStream_t)stream);
}
