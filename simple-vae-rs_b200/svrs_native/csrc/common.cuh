// common.cuh - shared helpers for the svrs_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../../include/svrs_b200.h"

namespace svrs {

void set_error(const char* fmt, ...);

#define SVRS_CHECK_ARG(cond, ...)                 \
    do {                                          \
        if (!(cond)) {                            \
            svrs::set_error(__VA_ARGS__);         \
            return SVRS_E_ARG;                    \
        }                                         \
    } while (0)

void note_kernel(const char* what);   // launch counter + optional name trace (layout.cu)

static inline int check_launch(const char* what) {
    note_kernel(what);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return SVRS_E_CUDA;
    }
    return 0;
}

// ---- programmatic dependent launch (PDL) ---------------------------------------------------------------------------
// Every kernel of the library can be launched with the programmatic-stream-serialization attribute and starts with
// pdl_trigger() (let the NEXT kernel of the stream begin launching: its CTAs become resident as ours retire) and
// pdl_wait() (block until the PREVIOUS kernel of the stream has completed and flushed) before it touches global memory.
// That hides the kernel-to-kernel launch latency of the ~300 mostly tiny launches of a step; the tensor-core kernels
// additionally run their barrier / TMEM / tensor-map prologue ahead of pdl_wait().  The attribute is only set with
// SVRS_PDL=1 (without it the device-side instructions are no-ops): measured neutral under CUDA-graph replay.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_entry() { pdl_trigger(); pdl_wait(); }
bool pdl_enabled();   // layout.cu

template <typename... KArgs, typename... Args>
static inline void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#define SVRS_LAUNCH(kernel, grid, block, smem, st, ...) svrs::launch_k(kernel, dim3(grid), dim3(block), (size_t)(smem), st, __VA_ARGS__)

// NULL or 16-byte aligned: the condition for the float4 / uint4 accesses of the streaming kernels
static inline bool al16(const void* p) { return p == nullptr || ((uintptr_t)p & 15) == 0; }

static inline int num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

template <typename T> struct Cvt;
template <> struct Cvt<float> {
    __device__ __forceinline__ static float to_f(float v) { return v; }
    __device__ __forceinline__ static float from_f(float v) { return v; }
};
template <> struct Cvt<__nv_bfloat16> {
    __device__ __forceinline__ static float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
    __device__ __forceinline__ static __nv_bfloat16 from_f(float v) { return __float2bfloat16_rn(v); }
};

// 4-element vector load/store with dtype conversion to fp32.  `p` must be 4-element aligned.
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ld4(const __nv_bfloat16* p) {
    uint2 r = *reinterpret_cast<const uint2*>(p);
    __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&r.x);
    __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&r.y);
    float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
    return make_float4(fa.x, fa.y, fb.x, fb.y);
}
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4(__nv_bfloat16* p, float4 v) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y);
    __nv_bfloat162 b = __floats2bfloat162_rn(v.z, v.w);
    uint2 r;
    r.x = *reinterpret_cast<uint32_t*>(&a);
    r.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(p) = r;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ float apply_act(float v, int act) {
    if (act == SVRS_ACT_SIGMOID) return 1.0f / (1.0f + expf(-v));
    if (act == SVRS_ACT_HARDTANH7) return fminf(fmaxf(v, -7.0f), 7.0f);
    return v;
}

}  // namespace svrs
