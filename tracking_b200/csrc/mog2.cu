// K-MOG2: cv::BackgroundSubtractorMOG2::operator() + getBackgroundImage + threshold, fused.
//
// Replaces (reference tree):
//   MixtureOfGaussianV2BGS::process   package_bgs/MixtureOfGaussianV2BGS.cpp:56 (mog(in, fg, alpha)),
//                                     :59 (getBackgroundImage), :61-62 (threshold)
// whose arithmetic is OpenCV's modules/video/src/bgfg_gaussmix2.cpp (un-vendored dependency,
// member `mog` at package_bgs/MixtureOfGaussianV2BGS.h:30); spec = SURVEY.md Appendix A.4.
//
// Data layout in HBM (structure of arrays, per camera stream):
//   state  : tiles of 64 pixels x 25 fp32 planes (kernels.h: mog2_tile_off), plane q = mode*5 +
//            {0 weight, 1 variance, 2 muB, 3 muG, 4 muR}
//   nmodes : 1 u8 plane
//   = 101 B/px, read once and written once per launch (per T frames with temporal batching).
// A thread owns 4 consecutive pixels: every plane access is one 128-bit load/store and a warp
// touches 512 contiguous bytes per plane.  All per-pixel state (25 floats x 4 px) lives in
// registers; the mode loop, the weight-ordered insertion and the new-mode insertion are fully
// unrolled with compile-time register indices (no local memory).
//
// Planes of modes that are dead for all 4 pixels of a thread (m >= max nmodes) are neither loaded
// nor stored: the CPU reference does not touch them either, and the values are unobservable.
//
// Numerics: fp32, unfused (-fmad=false), IEEE division, strict left-to-right evaluation -- the
// kernel is bit-exact against OpenCV's CPU implementation (tests/test_mog2_parity.py).
#include "common.cuh"
#include "kernels.h"
#include "mog2_pixel.cuh"

namespace bgsb {

constexpr int PX = 4;   // pixels per thread

__device__ __forceinline__ float &f4c(float4 &v, int j)
{
    return j == 0 ? v.x : j == 1 ? v.y : j == 2 ? v.z : v.w;
}

template <bool SHADOWS>
__global__ void __launch_bounds__(128)
mog2_kernel(const __grid_constant__ Mog2Launch L)
{
    pdl_entry();
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long px0 = g * PX;
    if (px0 >= L.npx) return;
    const int s = blockIdx.y;
    float *state = L.state + (size_t)s * MOG2_PLANES * L.pstride + mog2_tile_off((size_t)px0);   // 4 | 64: one tile
    uint8_t *nmp = L.nmodes + (size_t)s * L.pstride + px0;
    const uint8_t *frames = L.frames + (size_t)s * L.T * L.npx * 3;
    uint8_t *fg = L.fg + (size_t)s * L.T * L.npx;
    uint8_t *bgout = L.bg ? L.bg + (size_t)s * (L.bg_last_only ? 1 : L.T) * L.npx * 3 : nullptr;
    const bool full = (px0 + PX <= L.npx);     // planes are padded to 32 px, frames are not

    // ---- load state (read once per launch) ----
    int n[PX];
    unsigned nm4 = L.fresh ? 0u : ld_stream_u32(nmp);
#pragma unroll
    for (int j = 0; j < PX; j++) n[j] = (nm4 >> (8 * j)) & 0xff;
    int nmax = max(max(n[0], n[1]), max(n[2], n[3]));

    float4 P[MOG2_PLANES];
#pragma unroll
    for (int m = 0; m < K; m++) {
        if (m < nmax) {
#pragma unroll
            for (int f = 0; f < 5; f++) P[m * 5 + f] = ld_stream_f4(state + (m * 5 + f) * MOG2_TILE);
        } else {
#pragma unroll
            for (int f = 0; f < 5; f++) P[m * 5 + f] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }

    for (int t = 0; t < L.T; t++) {
        // ---- this frame's 4 pixels: 12 bytes ----
        const uint8_t *fr = frames + (size_t)t * L.npx * 3 + px0 * 3;
        unsigned iw[3];
        if (full && (reinterpret_cast<uintptr_t>(fr) & 3) == 0) {
            iw[0] = ld_stream_u32(fr); iw[1] = ld_stream_u32(fr + 4); iw[2] = ld_stream_u32(fr + 8);
        } else {
#pragma unroll
            for (int i = 0; i < 3; i++) {
                unsigned v = 0;
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (px0 * 3 + i * 4 + k < (long long)L.npx * 3) v |= (unsigned)fr[i * 4 + k] << (8 * k);
                iw[i] = v;
            }
        }
        const float aT = L.alphaT[t], a1 = L.alpha1[t], prune = L.prune[t];
        const bool want_bg = bgout && (!L.bg_last_only || t == L.T - 1);

        unsigned mask4 = 0, ow[3] = {0, 0, 0};
#pragma unroll
        for (int j = 0; j < PX; j++) {
            Mode md[K];
#pragma unroll
            for (int m = 0; m < K; m++) {
                md[m].w = f4c(P[m * 5 + 0], j); md[m].v = f4c(P[m * 5 + 1], j);
                md[m].b = f4c(P[m * 5 + 2], j); md[m].g = f4c(P[m * 5 + 3], j); md[m].r = f4c(P[m * 5 + 4], j);
            }
            const int b0 = 3 * j, b1 = 3 * j + 1, b2 = 3 * j + 2;
            float x0 = (float)byte_of(iw[b0 >> 2], b0 & 3);
            float x1 = (float)byte_of(iw[b1 >> 2], b1 & 3);
            float x2 = (float)byte_of(iw[b2 >> 2], b2 & 3);
            unsigned bB = 0, bG = 0, bR = 0;
            unsigned raw = mog2_pixel<SHADOWS>(md, n[j], x0, x1, x2, aT, a1, prune, L, bB, bG, bR, want_bg);
            mask4 |= thr_u8(raw, L.enable_thr, L.thr) << (8 * j);      // MixtureOfGaussianV2BGS.cpp:61-62
            ow[b0 >> 2] |= bB << (8 * (b0 & 3));
            ow[b1 >> 2] |= bG << (8 * (b1 & 3));
            ow[b2 >> 2] |= bR << (8 * (b2 & 3));
#pragma unroll
            for (int m = 0; m < K; m++) {
                f4c(P[m * 5 + 0], j) = md[m].w; f4c(P[m * 5 + 1], j) = md[m].v;
                f4c(P[m * 5 + 2], j) = md[m].b; f4c(P[m * 5 + 3], j) = md[m].g; f4c(P[m * 5 + 4], j) = md[m].r;
            }
        }

        // ---- per-frame outputs ----
        uint8_t *fgp = fg + (size_t)t * L.npx + px0;
        if (full && (reinterpret_cast<uintptr_t>(fgp) & 3) == 0) st_stream_u32(fgp, mask4);
        else {
#pragma unroll
            for (int j = 0; j < PX; j++) if (px0 + j < L.npx) fgp[j] = (uint8_t)(mask4 >> (8 * j));
        }
        if (want_bg) {
            uint8_t *bp = bgout + (L.bg_last_only ? 0 : (size_t)t * L.npx * 3) + px0 * 3;
            if (full && (reinterpret_cast<uintptr_t>(bp) & 3) == 0) { st_stream_u32(bp, ow[0]); st_stream_u32(bp + 4, ow[1]); st_stream_u32(bp + 8, ow[2]); }
            else {
#pragma unroll
                for (int i = 0; i < 12; i++)
                    if (px0 * 3 + i < (long long)L.npx * 3) bp[i] = (uint8_t)(ow[i >> 2] >> (8 * (i & 3)));
            }
        }
    }

    // ---- store state (written once per launch) ----
    int nmax2 = max(max(n[0], n[1]), max(n[2], n[3]));
#pragma unroll
    for (int m = 0; m < K; m++) {
        if (m < nmax2) {
#pragma unroll
            for (int f = 0; f < 5; f++) st_stream_f4(state + (m * 5 + f) * MOG2_TILE, P[m * 5 + f]);
        }
    }
    st_stream_u32(nmp, (unsigned)n[0] | ((unsigned)n[1] << 8) | ((unsigned)n[2] << 16) | ((unsigned)n[3] << 24));
}

int launch_mog2_t1(const Mog2Launch &L, int nstreams, cudaStream_t stream);
int launch_mog2_fused(const Mog2Launch &L, int nstreams, cudaStream_t stream);

// variant: 0 production (T == 1: two-phase kernel; T > 1: temporal-fusion kernel; csrc/mog2_t1.cu)
//          1 straight restatement (this file) -- the reference point of profiles/r1_mog2_kernel_history.md
int launch_mog2(const Mog2Launch &L, int nstreams, int variant, cudaStream_t stream)
{
    if (variant == 0) return L.T == 1 ? launch_mog2_t1(L, nstreams, stream) : launch_mog2_fused(L, nstreams, stream);
    const int threads = 128;
    long long nthreads = ((long long)L.npx + PX - 1) / PX;
    dim3 grid((unsigned)((nthreads + threads - 1) / threads), (unsigned)nstreams);
    // the shadow test only changes the output when 127 survives the wrapper's threshold
    const bool shadows = L.detect_shadows && !(L.enable_thr && (L.thr < L.shadow_value || L.thr >= 255));
    if (shadows) launch_pdl(mog2_kernel<true>, dim3(grid), dim3(threads), 0, stream, L);
    else launch_pdl(mog2_kernel<false>, dim3(grid), dim3(threads), 0, stream, L);
    BGSB_LAUNCH_CHECK();
    return BGSB_OK;
}

}  // namespace bgsb
