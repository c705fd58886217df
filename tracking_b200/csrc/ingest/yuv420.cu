// Ingest stage: YUV 4:2:0 camera frames (NV12: interleaved U,V; I420: planar U then V) to the dense BGR frames every
// plugin reads, as cv::cvtColor(COLOR_YUV2BGR_NV12 / COLOR_YUV2BGR_I420) computes them on 8-bit data: BT.601 limited
// range in 20-bit fixed point, each U,V pair shared by a 2x2 block of Y samples,
//
//     y = max(Y - 16, 0) * CY;  u = U - 128;  v = V - 128
//     B = sat_u8((y + 2^19 + CUB * u) >> 20)
//     G = sat_u8((y + 2^19 + CVG * v + CUG * u) >> 20)
//     R = sat_u8((y + 2^19 + CVR * v) >> 20)
//
// Every intermediate fits an int32 (|y + 2^19 + CVG*v + CUG*u| < 2^30), and >> is the arithmetic shift.
//
// Bound: HBM, 1.5 B/px read and 3 B/px written.  One warp converts 512 pixels of two rows (one chroma row): a lane owns
// 16 pixels x 2 rows and reads them as two 128-bit Y loads plus one 128-bit (NV12) or two 64-bit (I420) chroma loads.
// Its 2 x 48 BGR bytes go to the warp's shared-memory span first, and the warp stores each row's span as aligned,
// consecutive 128-bit chunks (a lane-strided 48-byte store pattern would make every 128-bit store straddle two L2
// sectors).  Ragged widths, odd chroma pitches and unaligned caller pointers take a per-pixel path for the lanes they
// touch, and the span's unaligned head and tail are stored byte by byte: no byte outside the frame is read or written.
#include "../common.cuh"
#include "../kernels.h"

namespace bgsb {

namespace {

constexpr int CY = 1220542, CUB = 2116026, CUG = -409993, CVG = -852492, CVR = 1673527;
constexpr int SHIFT = 20, HALF = 1 << (SHIFT - 1);
constexpr int PX_PER_LANE = 16, PX_PER_WARP = 32 * PX_PER_LANE;
constexpr int SPAN = PX_PER_WARP * 3;                       // BGR bytes of one row of a warp
constexpr int SPAN_PAD = SPAN + 16;                         // the aligned reader looks one word past a full chunk
constexpr int WARPS = 8;

__device__ __forceinline__ unsigned sat8(int x) { return (unsigned)min(max(x, 0), 255); }

// The three chroma terms of one U,V pair (rounding constant included)
struct Chroma { int b, g, r; };
__device__ __forceinline__ Chroma chroma(unsigned U, unsigned V)
{
    const int u = (int)U - 128, v = (int)V - 128;
    return Chroma{HALF + CUB * u, HALF + CVG * v + CUG * u, HALF + CVR * v};
}

// B | G << 8 | R << 16 of one pixel
__device__ __forceinline__ unsigned bgr_px(unsigned Y, const Chroma &c)
{
    const int y = max((int)Y - 16, 0) * CY;
    return sat8((y + c.b) >> SHIFT) | sat8((y + c.g) >> SHIFT) << 8 | sat8((y + c.r) >> SHIFT) << 16;
}

// 16 pixels (three bytes each) as 12 little-endian words
__device__ __forceinline__ void pack16(const unsigned px[16], unsigned out[12])
{
#pragma unroll
    for (int k = 0; k < 4; k++) {             // 4 pixels -> 3 words
        const unsigned a = px[4 * k], b = px[4 * k + 1], c = px[4 * k + 2], d = px[4 * k + 3];
        out[3 * k] = a | b << 24;
        out[3 * k + 1] = b >> 8 | c << 16;
        out[3 * k + 2] = c >> 16 | d << 8;
    }
}

// Store `len` bytes of a warp's shared-memory span to dst (any alignment): the chunks of dst's aligned 16-byte grid
// that lie wholly inside the span as 128-bit stores, the partial first and last chunks byte by byte.
__device__ __forceinline__ void store_span(const unsigned char *sp, uint8_t *dst, int len, int lane)
{
    const int a = (int)((uintptr_t)dst & 15);
    uint8_t *const base = dst - a;
    const int nchunks = (a + len + 15) >> 4;
    const unsigned *const spw = reinterpret_cast<const unsigned *>(sp);
    for (int k = lane; k < nchunks; k += 32) {
        const int s = 16 * k - a;
        if (s >= 0 && s + 16 <= len) {
            const int q = s >> 2, sh = (s & 3) * 8;
            const unsigned w0 = spw[q], w1 = spw[q + 1], w2 = spw[q + 2], w3 = spw[q + 3], w4 = spw[q + 4];
            uint4 v;
            v.x = __funnelshift_r(w0, w1, sh); v.y = __funnelshift_r(w1, w2, sh);
            v.z = __funnelshift_r(w2, w3, sh); v.w = __funnelshift_r(w3, w4, sh);
            st_stream_u4(base + 16 * k, v);
        } else {
            for (int j = 0; j < 16; j++) {
                const int o = s + j;
                if (o >= 0 && o < len) base[16 * k + j] = sp[o];
            }
        }
    }
}

}  // namespace

// PLANAR = false: NV12 (u points at the interleaved U,V rows); true: I420 (u, v at the U and V planes).
// Work item = (frame, row pair, 512-pixel column block), one per warp.
template <bool PLANAR>
__global__ void __launch_bounds__(WARPS * 32) yuv420_to_bgr_kernel(const Yuv420Launch L, long long nitems, int xblocks)
{
    pdl_entry();
    __shared__ __align__(16) unsigned char span[WARPS][2][SPAN_PAD];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const long long item = (long long)blockIdx.x * WARPS + wid;
    if (item >= nitems) return;
    const int xb = (int)(item % xblocks);
    const long long rest = item / xblocks;
    const int pairs = L.rows >> 1;
    const int rp = (int)(rest % pairs);
    const long long f = rest / pairs;
    const int x0 = xb * PX_PER_WARP, x = x0 + lane * PX_PER_LANE;
    const int ncols = min(PX_PER_WARP, L.w - x0);

    const uint8_t *const y0 = L.y + f * L.src_frame_stride + (size_t)(2 * rp) * L.y_pitch;
    const uint8_t *const y1 = y0 + L.y_pitch;
    const uint8_t *const cu = L.u + f * L.src_frame_stride + (size_t)rp * L.c_pitch;
    const uint8_t *const cv = PLANAR ? L.v + f * L.src_frame_stride + (size_t)rp * L.c_pitch : nullptr;
    unsigned char(*const sp)[SPAN_PAD] = span[wid];

    if (x < L.w) {
        unsigned px0[16], px1[16];
        const bool vec = x + PX_PER_LANE <= L.w && ((uintptr_t)(y0 + x) & 15) == 0 && ((uintptr_t)(y1 + x) & 15) == 0 &&
                         (PLANAR ? (((uintptr_t)(cu + x / 2) | (uintptr_t)(cv + x / 2)) & 7) == 0
                                 : ((uintptr_t)(cu + x) & 15) == 0);
        if (vec) {
            const uint4 a = ld_stream_u4(y0 + x), b = ld_stream_u4(y1 + x);
            const unsigned ya[4] = {a.x, a.y, a.z, a.w}, yb[4] = {b.x, b.y, b.z, b.w};
            unsigned cw[4];                     // chroma of the 8 pairs: NV12 U,V interleaved; I420 U words then V words
            if (PLANAR) {
                const uint2 uu = *reinterpret_cast<const uint2 *>(cu + x / 2), vv = *reinterpret_cast<const uint2 *>(cv + x / 2);
                cw[0] = uu.x; cw[1] = uu.y; cw[2] = vv.x; cw[3] = vv.y;
            } else {
                const uint4 c = ld_stream_u4(cu + x);
                cw[0] = c.x; cw[1] = c.y; cw[2] = c.z; cw[3] = c.w;
            }
#pragma unroll
            for (int p = 0; p < 8; p++) {
                const unsigned U = PLANAR ? byte_of(cw[p >> 2], p & 3) : byte_of(cw[p >> 1], 2 * (p & 1));
                const unsigned V = PLANAR ? byte_of(cw[2 + (p >> 2)], p & 3) : byte_of(cw[p >> 1], 2 * (p & 1) + 1);
                const Chroma c = chroma(U, V);
#pragma unroll
                for (int e = 0; e < 2; e++) {
                    const int i = 2 * p + e;
                    px0[i] = bgr_px(byte_of(ya[i >> 2], i & 3), c);
                    px1[i] = bgr_px(byte_of(yb[i >> 2], i & 3), c);
                }
            }
        } else {
            // per pixel: ragged right edge, odd chroma pitch or unaligned rows (only bytes inside the frame are read)
#pragma unroll
            for (int i = 0; i < 16; i++) {
                px0[i] = px1[i] = 0;
                const int xi = x + i;
                if (xi < L.w) {
                    const int cx = xi >> 1;
                    const unsigned U = PLANAR ? cu[cx] : cu[2 * cx], V = PLANAR ? cv[cx] : cu[2 * cx + 1];
                    const Chroma c = chroma(U, V);
                    px0[i] = bgr_px(y0[xi], c);
                    px1[i] = bgr_px(y1[xi], c);
                }
            }
        }
        unsigned o0[12], o1[12];
        pack16(px0, o0);
        pack16(px1, o1);
        uint4 *const s0 = reinterpret_cast<uint4 *>(sp[0] + 48 * lane), *const s1 = reinterpret_cast<uint4 *>(sp[1] + 48 * lane);
#pragma unroll
        for (int k = 0; k < 3; k++) {
            s0[k] = make_uint4(o0[4 * k], o0[4 * k + 1], o0[4 * k + 2], o0[4 * k + 3]);
            s1[k] = make_uint4(o1[4 * k], o1[4 * k + 1], o1[4 * k + 2], o1[4 * k + 3]);
        }
    }
    __syncwarp();
    uint8_t *const d0 = L.bgr + f * L.dst_frame_stride + ((size_t)(2 * rp) * L.w + x0) * 3;
    store_span(sp[0], d0, ncols * 3, lane);
    store_span(sp[1], d0 + (size_t)L.w * 3, ncols * 3, lane);
}

int launch_yuv420_to_bgr(const Yuv420Launch &L, cudaStream_t stream)
{
    BGSB_REQUIRE(L.w > 0 && L.rows > 0 && L.w % 2 == 0 && L.rows % 2 == 0 && L.nframes >= 1, "YUV 4:2:0 needs even sizes");
    const int xblocks = (L.w + PX_PER_WARP - 1) / PX_PER_WARP;
    const long long nitems = (long long)L.nframes * (L.rows / 2) * xblocks;
    const long long nblocks = (nitems + WARPS - 1) / WARPS;
    BGSB_REQUIRE(nblocks < (1LL << 31), "frame set too large");
    if (L.planar) launch_pdl(yuv420_to_bgr_kernel<true>, dim3((unsigned)nblocks), dim3(WARPS * 32), 0, stream, L, nitems, xblocks);
    else launch_pdl(yuv420_to_bgr_kernel<false>, dim3((unsigned)nblocks), dim3(WARPS * 32), 0, stream, L, nitems, xblocks);
    BGSB_LAUNCH_CHECK();
    return BGSB_OK;
}

}  // namespace bgsb
