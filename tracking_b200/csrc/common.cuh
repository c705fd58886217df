// Shared device/host helpers for libbgsb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <atomic>

#include "../../include/bgsb200.h"

namespace bgsb {

// Number of SMs of `device` (148 on a B200: 2 dies x 74), queried once per device; persistent / cooperative grids are
// sized from it.  capi.cu
int sm_count(int device);

// ---- error plumbing --------------------------------------------------------------------
void set_error(const char *fmt, ...);
extern std::atomic<uint64_t> g_launches;

#define BGSB_CUDA(call)                                                                      \
    do {                                                                                     \
        cudaError_t _e = (call);                                                             \
        if (_e != cudaSuccess) {                                                             \
            bgsb::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
            return BGSB_ERR_CUDA;                                                            \
        }                                                                                    \
    } while (0)

// launch_pdl() parks the status cudaLaunchKernelEx returned here; BGSB_LAUNCH_CHECK reads it first, so a failed launch is
// reported by the call that made it even when the error is not sticky in the runtime's per-thread state.
inline thread_local cudaError_t g_launch_status = cudaSuccess;

#define BGSB_LAUNCH_CHECK()                                                                  \
    do {                                                                                     \
        bgsb::g_launches.fetch_add(1, std::memory_order_relaxed);                            \
        cudaError_t _e = bgsb::g_launch_status;                                              \
        bgsb::g_launch_status = cudaSuccess;                                                 \
        if (_e == cudaSuccess) _e = cudaGetLastError(); else (void)cudaGetLastError();       \
        if (_e != cudaSuccess) {                                                             \
            bgsb::set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return BGSB_ERR_CUDA;                                                            \
        }                                                                                    \
    } while (0)

// ---- programmatic dependent launch -----------------------------------------------------------------
// Every kernel of the library is launched with the programmatic-stream-serialization attribute and starts with
// pdl_entry(): its grid may become resident while the previous kernel of the stream drains, and waits there
// until that kernel has completed and flushed.  This hides the launch ramp between the small dependent kernels
// of a stream (one MOG2 kernel per frame, the 12-kernel labelling chain).  Rules: pdl_entry() is the first
// statement, executed by every thread before any memory access or exit -- a grid whose CTAs left without waiting
// would complete early and release ITS successor before the predecessor's data is visible.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_entry()
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

template <typename... KArgs, typename... Args>
inline void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args &&... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
    if (e != cudaSuccess && g_launch_status == cudaSuccess) g_launch_status = e;     // reported by BGSB_LAUNCH_CHECK
}
#endif

#define BGSB_REQUIRE(cond, msg)                                                              \
    do {                                                                                     \
        if (!(cond)) {                                                                       \
            bgsb::set_error("%s: %s", __func__, msg);                                        \
            return BGSB_ERR_ARG;                                                             \
        }                                                                                    \
    } while (0)

// ---- per-pixel scalar pieces shared by the plugins ------------------------------------------
// cv::cvtColor(CV_BGR2GRAY) on 8-bit data (reference call sites FrameDifferenceBGS.cpp:48,
// AdaptiveBackgroundLearning.cpp:68, WeightedMovingVarianceBGS.cpp:103).  VARIANT 0 = OpenCV 4.x
// 15-bit coefficients, 1 = OpenCV 2.4 14-bit coefficients (SURVEY Appendix B).
template <int VARIANT>
__device__ __forceinline__ unsigned gray_bgr(unsigned b, unsigned g, unsigned r)
{
    if (VARIANT == 0) return (3735u * b + 19235u * g + 9798u * r + 16384u) >> 15;
    return (1868u * b + 9617u * g + 4899u * r + 8192u) >> 14;
}

// The same value from a pixel's three bytes packed B | G << 8 | R << 16 (the fourth byte is ignored): the 15- / 14-bit
// coefficients split into two bytes each, so the weighted sum is two 4-way byte dot products (IDP.4A) and a shift-add
// instead of three extractions and three multiply-adds -- the same integers, the same result.
template <int VARIANT>
__device__ __forceinline__ unsigned gray_px(unsigned px)
{
    if (VARIANT == 0) {                 // 3735 = 14 * 256 + 151, 19235 = 75 * 256 + 35, 9798 = 38 * 256 + 70
        const unsigned lo = __dp4a(px, 0x00462397u, 16384u), hi = __dp4a(px, 0x00264b0eu, 0u);
        return ((hi << 8) + lo) >> 15;
    }
    const unsigned lo = __dp4a(px, 0x0023914cu, 8192u), hi = __dp4a(px, 0x00132507u, 0u);      // 1868, 9617, 4899
    return ((hi << 8) + lo) >> 14;
}

// cv::threshold(..., THRESH_BINARY): strict '>' ; thr < 0 encodes enableThreshold == false
// only where the caller says so (see kernels).
__device__ __forceinline__ unsigned thr_u8(unsigned v, int enable, int thr)
{
    return enable ? (((int)v > thr) ? 255u : 0u) : v;
}

// saturate_cast<uchar>(float) = cvRound (round half to even) + clamp
__device__ __forceinline__ unsigned sat_u8_rint(float x)
{
    float r = rintf(x);
    r = fminf(fmaxf(r, 0.f), 255.f);   // NaN -> 0 via fmaxf
    return (unsigned)r;
}

// ---- streaming loads / stores ----------------------------------------------------------------
// State and frames are touched exactly once per launch: keep them out of L1
// (L2 eviction-priority qualifiers are only accepted on 256-bit loads by ptxas 12.9).
__device__ __forceinline__ float4 ld_stream_f4(const float *p)
{
    float4 v;
    asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_stream_f4(float *p, float4 v)
{
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ uint4 ld_stream_u4(const void *p)
{
    uint4 v;
    asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_stream_u4(void *p, uint4 v)
{
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ unsigned ld_stream_u32(const void *p)
{
    unsigned v;
    asm volatile("ld.global.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_stream_u32(void *p, unsigned v)
{
    asm volatile("st.global.L1::no_allocate.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}

__device__ __forceinline__ unsigned byte_of(unsigned word, int i) { return (word >> (8 * i)) & 0xffu; }

}  // namespace bgsb
