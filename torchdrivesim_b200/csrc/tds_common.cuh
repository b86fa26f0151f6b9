// Shared helpers for libtds_b200 (sm_100a).  The library is compiled with -fmad=false: every
// fp32 multiply/add is separately rounded, which is what the reference's eager torch CPU ops do
// (checked bit-for-bit in the build container), so oracle and kernels agree to the last bit
// wherever the transcendental inputs agree.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/tds_b200.h"

namespace tds {

std::string& last_error();
int fail(int code, const char* fmt, ...);
int sm_count();

#define TDS_REQUIRE(cond, ...)                                            \
    do {                                                                  \
        if (!(cond)) return ::tds::fail(TDS_ERR_INVALID_ARGUMENT, __VA_ARGS__); \
    } while (0)

#define TDS_CUDA_OK(expr)                                                                 \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess)                                                            \
            return ::tds::fail(TDS_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(_e)); \
    } while (0)

#define TDS_LAUNCH_OK()                                                                   \
    do {                                                                                  \
        cudaError_t _e = cudaGetLastError();                                              \
        if (_e != cudaSuccess)                                                            \
            return ::tds::fail(TDS_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(_e)); \
    } while (0)

// A launch with more than 48 KB of dynamic shared memory fails unless the kernel opts in first.
template <class K>
int allow_dynamic_smem(K kernel, size_t bytes) {
    if (bytes > 48 * 1024) TDS_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return TDS_OK;
}

// sin/cos evaluated in double and rounded to fp32: effectively correctly rounded, hence
// reproducible on the CPU (the oracle does the same) and within 1 ulp of torch's CPU sin/cos.
__device__ __forceinline__ void sincos_cr(float a, float& s, float& c) {
    double ds, dc;
    sincos((double)a, &ds, &dc);
    s = (float)ds;
    c = (float)dc;
}

// Corner k of the box (x, y, length l, width w) with heading sincos (s, c), in the corner order of box2corners_th
// (_iou_utils.py:270-299): (+,+), (-,+), (-,-), (+,-) half-extents rotated by psi.  The offroad and range-scan kernels
// share this arithmetic, so their corners agree bit for bit.
__device__ __forceinline__ void box_corner(float x, float y, float l, float w, float s, float c, int k, float& px, float& py) {
    const float sx = (k == 0 || k == 3) ? 0.5f : -0.5f;
    const float sy = (k < 2) ? 0.5f : -0.5f;
    const float ux = sx * l, uy = sy * w;
    px = (ux * c + uy * (-s)) + x;
    py = (ux * s + uy * c) + y;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// streaming 128-bit store: the image is written once and never re-read by this kernel
__device__ __forceinline__ void st_cs_f4(float4* p, float4 v) {
    asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}

__device__ __forceinline__ void st_cs_u32(uint32_t* p, uint32_t v) {
    asm volatile("st.global.cs.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

}  // namespace tds
