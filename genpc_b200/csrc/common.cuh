// common.cuh -- shared device helpers for libgenpc_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/genpc_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libgenpc_b200 is written for sm_100a (B200) only"
#endif

#define GENPC_NUM_SMS_B200 148   // compile-time sizes only (fixed-size reduction grids); launch shaping asks the device

namespace genpc {
// SMs of the CURRENT device (cached per device ordinal; tunables.cu).  B200: 148.  Grid sizes and the balanced / persistent
// heuristics use this, so a part with fewer SMs or a process driving several different devices is tuned correctly.
int num_sms();
}  // namespace genpc
#define GENPC_NUM_SMS (genpc::num_sms())

namespace genpc {

// Experiment knob `name` (GENPC_*): its value as read from the environment when the library was loaded or as set through
// genpc_set_tunable(); nullptr when unset.  Never calls getenv() (tunables.cu).
const char *tunable(const char *name);

// Lays out a workspace region by region.  Without a base, take() only adds up the bytes, so ONE function per workspace both
// sizes it and carves it.  Alignments are offsets from the base, except after align_base().
struct WsCursor {
    char *base;   // nullptr: sizing only
    size_t off = 0, before = 0;
    template <typename T>
    T *take(size_t count, size_t align = alignof(T)) {
        off = (off + align - 1) / align * align;
        T *p = base != nullptr ? reinterpret_cast<T *>(base + off) : nullptr;
        off += count * sizeof(T);
        return p;
    }
    // Continue at the next 256-byte boundary of the address.  The size reserves the worst-case pad of 255 bytes, so it is
    // exact whatever the base; later alignments are offsets from the boundary.
    void align_base() {
        if (base != nullptr) base += off + (256 - reinterpret_cast<size_t>(base + off) % 256) % 256;
        before += off + 255, off = 0;
    }
    size_t bytes() const { return before + off; }
};

// Programmatic dependent launch: kernel<<<grid, block, 0, stream>>>(args...) may be dispatched while the kernel before it on
// `stream` is still draining (from the moment every CTA of that kernel has called cudaTriggerProgrammaticLaunchCompletion()
// or exited), so the launch latency between two of the library's kernels overlaps the first one's tail.  A kernel launched
// this way calls cudaGridDependencySynchronize() in every CTA before it touches global memory that an earlier launch on the
// stream reads or writes (and before it can exit, so that its own completion still implies its predecessor's); only parameter
// decoding and index math come first.
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid, cfg.blockDim = block, cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr, cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, args...);
}

// The whole library is compiled with -fmad=false: every contraction below is explicit, because the
// reference's indices depend on the exact rounding order (SURVEY.md section 2b).

// 3-input float min (FMNMX3 on sm_100a); NaN operands are ignored (IEEE minNum).
__device__ __forceinline__ float fmin3(float a, float b, float c) {
    float r;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}

// Squared distance with the reference's rounding order (chamfer3D.cu:35 under -fmad=true):
// d = fma(dz,dz, fma(dx,dx, dy*dy)), d* = target - query.
__device__ __forceinline__ float sqdist_ref(float qx, float qy, float qz, float tx, float ty, float tz) {
    float dx = __fsub_rn(tx, qx), dy = __fsub_rn(ty, qy), dz = __fsub_rn(tz, qz);
    return __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
}

// Two targets at once on the packed FP32 pipe (FADD2 / FMUL2 / FFMA2, new on sm_100).
// nq* hold the NEGATED query coordinate duplicated in both halves; t* hold (target_k, target_k+1).
// t + (-q) == t - q exactly, so each half is bit-identical to sqdist_ref.
__device__ __forceinline__ float2 sqdist_ref_x2(float2 nqx, float2 nqy, float2 nqz, float2 tx, float2 ty,
                                                float2 tz) {
    float2 dx = __fadd2_rn(tx, nqx);
    float2 dy = __fadd2_rn(ty, nqy);
    float2 dz = __fadd2_rn(tz, nqz);
    float2 s = __fmul2_rn(dy, dy);
    s = __ffma2_rn(dx, dx, s);
    s = __ffma2_rn(dz, dz, s);
    return s;
}

// (dist, idx) packed so that unsigned 64-bit order == (dist ascending, idx ascending).
// dist is a sum of squares => non-negative => its bit pattern orders like the float.
__device__ __forceinline__ unsigned long long pack_dist_idx(float d, int idx) {
    return ((unsigned long long)__float_as_uint(d) << 32) | (unsigned int)idx;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace genpc

#define GENPC_CHECK_LAUNCH()                         \
    do {                                             \
        cudaError_t e__ = cudaGetLastError();        \
        if (e__ != cudaSuccess) return (int)e__;     \
    } while (0)
