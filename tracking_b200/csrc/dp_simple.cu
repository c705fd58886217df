// K-DPS: the three simple per-pixel models of the reference's DP package (sibling plugins, SURVEY 8f N3 widened):
//
//   DPAdaptiveMedianBGS  USTC_BGS type 9   package_bgs/dp/AdaptiveMedianBGS.cpp:53-140   (wrapper DPAdaptiveMedianBGS.cpp:28-82)
//   DPMeanBGS            USTC_BGS type 12  package_bgs/dp/MeanBGS.cpp:32-131            (wrapper DPMeanBGS.cpp:28-84)
//   DPWrenGABGS          USTC_BGS type 13  package_bgs/dp/WrenGA.cpp:47-173             (wrapper DPWrenGABGS.cpp:28-84)
//
// Every wrapper does, per frame: Subtract (mask from the CURRENT model; the plugin's output is the HIGH-threshold mask),
// clear the low mask, Update on every pixel (the cleared mask makes the learning-frames test vacuous).  img_bgmodel is
// never written.  The reference makes two full passes with per-pixel accessor calls; here one thread owns 4 pixels
// (12 frame bytes = three words), reads the model once, writes mask and model once:
//   AdaptiveMedian  3 in + 3 model + 1 mask (+ 3 model on the frames whose number is 1 modulo samplingRate)  =  7 / 10 B/px
//   Mean            3 in + 12 mean read + 12 written + 1 mask                                                = 28 B/px
//   WrenGA          3 in + 16 (mu, var) read + 16 written + 1 mask                                           = 36 B/px
// fp32 arithmetic in the reference's order, unfused (the library is compiled with -fmad=false; the operations are
// written with the _rn intrinsics anyway).  Parity: bit-exact against the CPU restatement, which is pinned to a build of
// the reference's own sources (tests/golden/golden_dp.json, tests/test_oracle_pin.py).
#include <stdlib.h>
#include <initializer_list>
#include "common.cuh"
#include "kernels.h"

namespace bgsb {

// the 12 bytes of 4 pixels as three words (B0 G0 R0 B1 | G1 R1 B2 G2 | R2 B3 G3 R3); `n` valid pixels, zero fill
__device__ __forceinline__ void dps_load12(const uint8_t *p, bool vec, int n, unsigned (&w)[3])
{
    if (vec) {
        const unsigned *q = reinterpret_cast<const unsigned *>(p);
        w[0] = ld_stream_u32(q); w[1] = ld_stream_u32(q + 1); w[2] = ld_stream_u32(q + 2);
    } else {
        w[0] = w[1] = w[2] = 0u;
        for (int i = 0; i < 3 * n; i++) w[i >> 2] |= (unsigned)p[i] << (8 * (i & 3));
    }
}
__device__ __forceinline__ void dps_store12(uint8_t *p, bool vec, int n, const unsigned (&w)[3])
{
    if (vec) {
        unsigned *q = reinterpret_cast<unsigned *>(p);
        st_stream_u32(q, w[0]); st_stream_u32(q + 1, w[1]); st_stream_u32(q + 2, w[2]);
    } else {
        for (int i = 0; i < 3 * n; i++) p[i] = (uint8_t)(w[i >> 2] >> (8 * (i & 3)));
    }
}
__device__ __forceinline__ void dps_store_mask(uint8_t *p, bool vec, int n, unsigned m)
{
    if (vec) st_stream_u32(p, m);
    else for (int i = 0; i < n; i++) p[i] = (uint8_t)(m >> (8 * i));
}
__device__ __forceinline__ unsigned dps_byte(const unsigned (&w)[3], int i) { return (w[i >> 2] >> (8 * (i & 3))) & 0xffu; }

__global__ void __launch_bounds__(256)
dps_median_kernel(DpsLaunch L)
{
    pdl_entry();
    const long long px0 = ((long long)blockIdx.x * 256 + threadIdx.x) * 4;
    if (px0 >= L.npx) return;
    const int n = (int)min(4LL, (long long)L.npx - px0);
    const size_t s = blockIdx.y;
    const uint8_t *fp = L.frame + s * L.frame_stride + px0 * 3;
    uint8_t *mp = L.median + s * L.median_stride + px0 * 3;
    uint8_t *gp = L.fg + s * L.fg_stride + px0;
    const bool v12 = n == 4 && ((reinterpret_cast<uintptr_t>(fp) | reinterpret_cast<uintptr_t>(mp)) & 3) == 0;
    const bool v4 = n == 4 && (reinterpret_cast<uintptr_t>(gp) & 3) == 0;
    unsigned in[3], med[3];
    dps_load12(fp, v12, n, in);
    if (L.fresh) { med[0] = in[0]; med[1] = in[1]; med[2] = in[2]; }           // InitModel :53-63
    else dps_load12(mp, v12, n, med);
    // SubtractPixel :92-111: foreground unless all three |pixel - median| <= high
    const unsigned hi = L.high_u * 0x01010101u;
    unsigned gt[3];
#pragma unroll
    for (int k = 0; k < 3; k++) gt[k] = __vcmpgtu4(__vabsdiffu4(in[k], med[k]), hi) & 0x01010101u;
    const unsigned p0 = gt[0] & 0x00ffffffu, p1 = __byte_perm(gt[0], gt[1], 0x0543u) & 0x00ffffffu;
    const unsigned p2 = __byte_perm(gt[1], gt[2], 0x0432u) & 0x00ffffffu, p3 = gt[2] >> 8;
    const unsigned m = (p0 ? 0xffu : 0u) | (p1 ? 0xff00u : 0u) | (p2 ? 0xff0000u : 0u) | (p3 ? 0xff000000u : 0u);
    dps_store_mask(gp, v4, n, m);
    // Update :65-90 (every pixel: the wrapper clears the update mask): one step towards the pixel, per channel
    if (L.update) {
#pragma unroll
        for (int k = 0; k < 3; k++)
            med[k] = med[k] + (__vcmpgtu4(in[k], med[k]) & 0x01010101u) - (__vcmpltu4(in[k], med[k]) & 0x01010101u);   // no byte carries
    }
    if (L.update || L.fresh) dps_store12(mp, v12, n, med);
}

// one pixel of MeanBGS / WrenGA: x = its three bytes as floats, m = its model (Mean: 3 means; WrenGA: 3 means + variance)
template <int KIND>
__device__ __forceinline__ unsigned dps_float_pixel(const DpsLaunch &L, const float (&x)[3], float (&m)[4])
{
    if (L.fresh) {                                       // InitModel (MeanBGS.cpp:40-52, WrenGA.cpp:67-85)
        m[0] = x[0]; m[1] = x[1]; m[2] = x[2];
        if (KIND == DPS_WREN) m[3] = 36.0f;
    }
    unsigned fg;
    if (KIND == DPS_MEAN) {
        float dist = 0.f;                                // SubtractPixel :77-99
#pragma unroll
        for (int c = 0; c < 3; c++) { const float d = __fsub_rn(x[c], m[c]); dist = __fadd_rn(dist, __fmul_rn(d, d)); }
        fg = dist > L.high_f ? 255u : 0u;
#pragma unroll
        for (int c = 0; c < 3; c++)                      // Update :54-75
            m[c] = __fadd_rn(__fmul_rn(L.alpha, m[c]), __fmul_rn(L.one_minus_alpha, x[c]));
    } else {
        float d[3], dist = 0.f;                          // SubtractPixel :121-147
#pragma unroll
        for (int c = 0; c < 3; c++) { d[c] = __fsub_rn(m[c], x[c]); dist = __fadd_rn(dist, __fmul_rn(d[c], d[c])); }
        fg = dist > __fmul_rn(L.high_f, m[3]) ? 255u : 0u;
#pragma unroll
        for (int c = 0; c < 3; c++) m[c] = __fsub_rn(m[c], __fmul_rn(L.alpha, d[c]));           // Update :97-105
        const float sig = __fadd_rn(m[3], __fmul_rn(L.alpha, __fsub_rn(dist, m[3])));
        m[3] = sig < 4.f ? 4.f : (sig > 180.f ? 180.f : sig);                                   // 5 * m_variance
    }
    return fg;
}

template <int KIND>
__global__ void __launch_bounds__(256)
dps_float_kernel(DpsLaunch L)
{
    pdl_entry();
    constexpr int NP = KIND == DPS_MEAN ? 3 : 4;
    const long long px0 = ((long long)blockIdx.x * 256 + threadIdx.x) * 4;
    if (px0 >= L.npx) return;
    const int n = (int)min(4LL, (long long)L.npx - px0);
    const size_t s = blockIdx.y;
    const uint8_t *fp = L.frame + s * L.frame_stride + px0 * 3;
    uint8_t *gp = L.fg + s * L.fg_stride + px0;
    float *st = L.state + s * NP * L.pstride + px0;      // plane q: st + q * pstride
    const bool v12 = n == 4 && (reinterpret_cast<uintptr_t>(fp) & 3) == 0;
    const bool v4 = n == 4 && (reinterpret_cast<uintptr_t>(gp) & 3) == 0;
    const bool v16 = n == 4 && (reinterpret_cast<uintptr_t>(st) & 15) == 0 && (L.pstride & 3) == 0;
    unsigned in[3];
    dps_load12(fp, v12, n, in);
    float pl[NP][4];
#pragma unroll
    for (int q = 0; q < NP; q++) {
        if (L.fresh) { pl[q][0] = pl[q][1] = pl[q][2] = pl[q][3] = 0.f; }
        else if (v16) { const float4 v = ld_stream_f4(st + q * L.pstride); pl[q][0] = v.x; pl[q][1] = v.y; pl[q][2] = v.z; pl[q][3] = v.w; }
        else {
#pragma unroll
            for (int j = 0; j < 4; j++) pl[q][j] = j < n ? st[q * L.pstride + j] : 0.f;
        }
    }
    unsigned m = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        float x[3], mod[4];
#pragma unroll
        for (int c = 0; c < 3; c++) x[c] = (float)dps_byte(in, 3 * j + c);
#pragma unroll
        for (int q = 0; q < NP; q++) mod[q] = pl[q][j];
        m |= dps_float_pixel<KIND>(L, x, mod) << (8 * j);
#pragma unroll
        for (int q = 0; q < NP; q++) pl[q][j] = mod[q];
    }
    dps_store_mask(gp, v4, n, m);
#pragma unroll
    for (int q = 0; q < NP; q++) {
        if (v16) st_stream_f4(st + q * L.pstride, make_float4(pl[q][0], pl[q][1], pl[q][2], pl[q][3]));
        else {
#pragma unroll
            for (int j = 0; j < 4; j++) if (j < n) st[q * L.pstride + j] = pl[q][j];
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// K-PRATI: DPPratiMediodBGS, USTC_BGS type 14 (package_bgs/dp/PratiMediodBGS.cpp:52-275, wrapper DPPratiMediodBGS.cpp:28-88).
// Pure integer.  The reference keeps, per pixel, std::vectors of up to H sampled pixels and of each sample's sum of L-inf
// distances to the others; the medoid (smallest sum, first wins) is the background.  The wrapper clears the update mask,
// so every pixel is sampled on the same frames: the per-pixel vectors are whole frames (samples[s]) and whole planes
// (dist[s], 16 bit: a sum never exceeds (H + 1) * 255), buffer length n and write position pos are host counters.
//   subtract (every frame >= H):  L-inf distance to the medoid against low / high threshold, then the hysteresis of
//       Combine(): high -> foreground; low -> foreground iff one of the 8 neighbours is high; image border -> background.
//       A thread owns 4 pixels; the neighbour test (rare: low-but-not-high pixels) recomputes the neighbours' distance.
//   update (frames with frame_num % samplingRate == 0):  one pass over the n samples per 4 pixels -- remove the replaced
//       sample's distances (ring full), add the new pixel's, track the medoid -- then the new pixel takes the slot.
//       The quirks are the reference's and are kept: the replaced sample still competes with its old sum, and the new
//       sample's sum includes its distance to the sample it replaces.
// ---------------------------------------------------------------------------------------------------------------
// Internal layout (ours, not the reference's): everything the model keeps is PLANAR in groups of 4 pixels -- a sample is
// three planes (B, G, R) of plane1 bytes, the medoid image likewise -- so that 4 pixels' channel values are one word per
// channel and the L-inf distance of 4 pixels is 3 byte-SIMD differences and two 3-way 16-bit SIMD maxima (VIMNMX3 on the
// even and on the odd bytes).  The distance sums are stored the way those maxima come out: per 4 pixels a uint2 whose
// .x holds pixels 0 and 2, .y pixels 1 and 3 (16 bits each), so sums, minima and comparisons stay packed too.
struct Planar4 { unsigned b, g, r; };
// 4 interleaved pixels (B0 G0 R0 B1 | G1 R1 B2 G2 | R2 B3 G3 R3) -> one word per channel
__device__ __forceinline__ Planar4 prati_planar(const unsigned (&w)[3])
{
    Planar4 p;
    p.b = __byte_perm(__byte_perm(w[0], w[1], 0x0630u), w[2], 0x5210u);
    p.g = __byte_perm(__byte_perm(w[0], w[1], 0x0741u), w[2], 0x6210u);
    p.r = __byte_perm(__byte_perm(w[0], w[1], 0x0052u), w[2], 0x7410u);
    return p;
}
// L-inf distances of 4 pixels: e = pixels 0 and 2, o = pixels 1 and 3 (16-bit lanes)
__device__ __forceinline__ void prati_linf4(const Planar4 &x, const Planar4 &y, unsigned &e, unsigned &o)
{
    const unsigned db = __vabsdiffu4(x.b, y.b), dg = __vabsdiffu4(x.g, y.g), dr = __vabsdiffu4(x.r, y.r);
    e = __vimax3_u16x2(db & 0x00ff00ffu, dg & 0x00ff00ffu, dr & 0x00ff00ffu);
    o = __vimax3_u16x2((db >> 8) & 0x00ff00ffu, (dg >> 8) & 0x00ff00ffu, (dr >> 8) & 0x00ff00ffu);
}
// byte mask (0xff per pixel) from the two lane masks (0xffff per 16-bit lane) of the even and the odd pixels
__device__ __forceinline__ unsigned prati_bytemask(unsigned me, unsigned mo) { return (me & 0x00ff00ffu) | (mo & 0xff00ff00u); }

__global__ void __launch_bounds__(256)
prati_subtract_kernel(PratiLaunch L)
{
    pdl_entry();
    const int npx = L.w * L.h;
    const long long px0 = ((long long)blockIdx.x * 256 + threadIdx.x) * 4;
    if (px0 >= npx) return;
    const int n = (int)min(4LL, (long long)npx - px0);
    const size_t s = blockIdx.y;
    const uint8_t *frame = L.frame + s * L.frame_stride;
    const uint8_t *median = L.state + s * L.stream_bytes + (size_t)L.H * L.plane3;      // planar: B, G, R planes of plane1 bytes
    uint8_t *gp = L.fg + s * L.fg_stride + px0;
    const uint8_t *fp = frame + px0 * 3;
    const bool v12 = n == 4 && (reinterpret_cast<uintptr_t>(fp) & 3) == 0;
    const bool v4 = n == 4 && (reinterpret_cast<uintptr_t>(gp) & 3) == 0;
    unsigned in[3];
    dps_load12(fp, v12, n, in);
    Planar4 med;
    med.b = *reinterpret_cast<const unsigned *>(median + px0);
    med.g = *reinterpret_cast<const unsigned *>(median + L.plane1 + px0);
    med.r = *reinterpret_cast<const unsigned *>(median + 2 * L.plane1 + px0);
    unsigned de, dodd;
    prati_linf4(prati_planar(in), med, de, dodd);                            // CalculateMasks :204-234
    const unsigned dist4[4] = {de & 0xffffu, dodd & 0xffffu, de >> 16, dodd >> 16};
    unsigned m = 0;
    const int r0 = (int)((unsigned)px0 / (unsigned)L.w), c0 = (int)((unsigned)px0 - (unsigned)r0 * (unsigned)L.w);      // 32-bit: frames hold < 2^30 pixels
#pragma unroll
    for (int j = 0; j < 4; j++) {
        if (j >= n) break;
        const unsigned dist = dist4[j];
        unsigned out = 0;
        int r = r0, c = c0 + j;
        while (c >= L.w) { c -= L.w; r++; }                                  // (widths below 4: a group spans several rows)
        const int p = (int)px0 + j;
        if (r > 0 && c > 0 && r < L.h - 1 && c < L.w - 1) {                 // Combine :167-202
            if (dist > L.high) out = 255u;
            else if (dist > L.low) {
                for (int dr = -1; dr <= 1 && !out; dr++)
                    for (int dc = -1; dc <= 1; dc++) {
                        if (!dr && !dc) continue;
                        const size_t qi = (size_t)(p + dr * L.w + dc), q = qi * 3;
                        const unsigned nd = max(max(__sad((int)frame[q], (int)median[qi], 0u),
                                                    __sad((int)frame[q + 1], (int)median[L.plane1 + qi], 0u)),
                                                __sad((int)frame[q + 2], (int)median[2 * L.plane1 + qi], 0u));
                        if (nd > L.high) { out = 255u; break; }
                    }
            }
        }
        m |= out << (8 * j);
    }
    dps_store_mask(gp, v4, n, m);
}

__global__ void __launch_bounds__(256)
prati_update_kernel(PratiLaunch L)
{
    pdl_entry();
    const int npx = L.w * L.h;
    const long long px0 = ((long long)blockIdx.x * 256 + threadIdx.x) * 4;
    if (px0 >= npx) return;
    const int n = (int)min(4LL, (long long)npx - px0);
    const size_t s = blockIdx.y;
    uint8_t *st = L.state + s * L.stream_bytes;
    uint8_t *samples = st + px0, *median = st + (size_t)L.H * L.plane3 + px0;
    uint2 *dist = reinterpret_cast<uint2 *>(st + (size_t)(L.H + 1) * L.plane3) + px0 / 4;      // plane k: + k * plane1 / 4
    const size_t dstride = L.plane1 / 4;
    const uint8_t *fp = L.frame + s * L.frame_stride + px0 * 3;
    const bool vin = n == 4 && (reinterpret_cast<uintptr_t>(fp) & 3) == 0;
    const bool full = L.n == L.H;
    unsigned in[3];
    dps_load12(fp, vin, n, in);                                             // ragged tail: zero fill; the planes are padded
    const Planar4 x = prati_planar(in);
    auto load_sample = [&](int k) {
        const uint8_t *p = samples + (size_t)k * L.plane3;
        Planar4 v;
        v.b = *reinterpret_cast<const unsigned *>(p);
        v.g = *reinterpret_cast<const unsigned *>(p + L.plane1);
        v.r = *reinterpret_cast<const unsigned *>(p + 2 * L.plane1);
        return v;
    };
    Planar4 old = {0u, 0u, 0u};
    if (full) old = load_sample(L.pos);
    unsigned best_e = 0xffffffffu, best_o = 0xffffffffu, sum_e = 0u, sum_o = 0u;       // best: INT_MAX stand-in per 16-bit lane
    Planar4 med = {0u, 0u, 0u};
    // sample k + 1 and its sums are requested before sample k is worked on
    Planar4 spn = {0u, 0u, 0u};
    uint2 dvn = make_uint2(0u, 0u);
    if (L.n > 0) { spn = load_sample(0); dvn = dist[0]; }
    for (int k = 0; k < L.n; k++) {
        const Planar4 sp = spn;
        uint2 ds = dvn;
        if (k + 1 < L.n) { spn = load_sample(k + 1); dvn = dist[(size_t)(k + 1) * dstride]; }
        unsigned ne, no;
        prati_linf4(sp, x, ne, no);
        if (full) {                                                         // Update :84-95
            unsigned oe, oo;
            prati_linf4(sp, old, oe, oo);
            ds.x -= oe; ds.y -= oo;                                         // per 16-bit lane: a sum holds every distance it loses
        }
        ds.x += ne; ds.y += no;                                             // UpdateMediod :143-155
        const unsigned bm = prati_bytemask(__vcmpltu2(ds.x, best_e), __vcmpltu2(ds.y, best_o));
        best_e = __vimin3_u16x2(best_e, ds.x, ds.x); best_o = __vimin3_u16x2(best_o, ds.y, ds.y);
        med.b = (sp.b & bm) | (med.b & ~bm); med.g = (sp.g & bm) | (med.g & ~bm); med.r = (sp.r & bm) | (med.r & ~bm);
        sum_e += ne; sum_o += no;
        dist[(size_t)k * dstride] = ds;
    }
    {   // the new point is the medoid :160-164
        const unsigned bm = prati_bytemask(__vcmpltu2(sum_e, best_e), __vcmpltu2(sum_o, best_o));
        med.b = (x.b & bm) | (med.b & ~bm); med.g = (x.g & bm) | (med.g & ~bm); med.r = (x.r & bm) | (med.r & ~bm);
    }
    *reinterpret_cast<unsigned *>(median) = med.b;
    *reinterpret_cast<unsigned *>(median + L.plane1) = med.g;
    *reinterpret_cast<unsigned *>(median + 2 * L.plane1) = med.r;
    // the new sample and its sum into the slot (:97-100 / :119-121)
    const int slot = full ? L.pos : L.n;
    uint8_t *sl = samples + (size_t)slot * L.plane3;
    *reinterpret_cast<unsigned *>(sl) = x.b;
    *reinterpret_cast<unsigned *>(sl + L.plane1) = x.g;
    *reinterpret_cast<unsigned *>(sl + 2 * L.plane1) = x.r;
    dist[(size_t)slot * dstride] = make_uint2(sum_e, sum_o);
}

int launch_prati_subtract(const PratiLaunch &L, int nstreams, cudaStream_t stream)
{
    const long long groups = ((long long)L.w * L.h + 3) / 4;
    launch_pdl(prati_subtract_kernel, dim3((unsigned)((groups + 255) / 256), (unsigned)nstreams), dim3(256), 0, stream, L);
    BGSB_LAUNCH_CHECK();
    return BGSB_OK;
}

int launch_prati_update(const PratiLaunch &L, int nstreams, cudaStream_t stream)
{
    const long long groups = ((long long)L.w * L.h + 3) / 4;
    launch_pdl(prati_update_kernel, dim3((unsigned)((groups + 255) / 256), (unsigned)nstreams), dim3(256), 0, stream, L);
    BGSB_LAUNCH_CHECK();
    return BGSB_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// K-SD: SigmaDeltaBGS, USTC_BGS type 35 (package_bgs/bl/sdLaMa091.cpp:117-232, :470-636; wrapper SigmaDeltaBGS.cpp:21-50).
// Pure integer and byte-wise, so 4 pixels = three words of byte-SIMD: the reference makes four passes over three images;
// here frame, Mt and Vt are read once and Mt, Vt and the mask written once (13 B/px).  Its byte-arithmetic quirks are kept:
// the difference passes through a signed char before the absolute value (|d| > 128 wraps), Vt steps in uint8_t (wraps when
// N > 1 pushes it past 255) and is clamped to the parameters truncated to a byte; the initialiser fills only the first
// `width` bytes of every row of Vt with Vmin (the rest is zero, see the oracle's notes).
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
sigma_delta_kernel(SdLaunch L)
{
    pdl_entry();
    const long long px0 = ((long long)blockIdx.x * 256 + threadIdx.x) * 4;
    if (px0 >= L.npx) return;
    const int n = (int)min(4LL, (long long)L.npx - px0);
    const size_t s = blockIdx.y;
    const uint8_t *fp = L.frame + s * L.frame_stride + px0 * 3;
    uint8_t *mp = L.Mt + s * L.model_stride + px0 * 3, *vp = L.Vt + s * L.model_stride + px0 * 3;
    uint8_t *gp = L.fg ? L.fg + s * L.fg_stride + px0 : nullptr;
    const bool v12 = n == 4 && ((reinterpret_cast<uintptr_t>(fp) | reinterpret_cast<uintptr_t>(mp) | reinterpret_cast<uintptr_t>(vp)) & 3) == 0;
    unsigned in[3], m[3], v[3];
    dps_load12(fp, v12, n, in);
    if (L.first) {                                                          // sdLaMa091AllocInit_8u_C3R -> _C1R (:155, :204-216)
        unsigned long long cb = (unsigned long long)((L.p0 + px0) * 3) % (unsigned long long)(3 * L.w);      // byte position inside the row
        v[0] = v[1] = v[2] = 0u;
        for (int i = 0; i < 12; i++) {
            if (cb < (unsigned long long)L.w) v[i >> 2] |= L.vmin8 << (8 * (i & 3));
            if (++cb == (unsigned long long)(3 * L.w)) cb = 0;
        }
        dps_store12(mp, v12, n, in);
        dps_store12(vp, v12, n, v);
        return;
    }
    dps_load12(mp, v12, n, m);
    dps_load12(vp, v12, n, v);
    const unsigned vmax4 = L.vmax8 * 0x01010101u, vmin4 = L.vmin8 * 0x01010101u;
    unsigned ge[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        m[k] = m[k] + (__vcmpltu4(m[k], in[k]) & 0x01010101u) - (__vcmpgtu4(m[k], in[k]) & 0x01010101u);      // :536-539 (no byte carries)
        const unsigned o = __vabs4(__vsub4(m[k], in[k]));                   // absVal((int8_t)(Mt - I)) :74-76, :559
        unsigned nv;
        if (L.N == 1u) nv = v[k] + (__vcmpltu4(v[k], o) & 0x01010101u) - (__vcmpgtu4(v[k], o) & 0x01010101u);  // :574-579
        else {
            nv = 0u;
#pragma unroll
            for (int b = 0; b < 4; b++) {
                unsigned vb = (v[k] >> (8 * b)) & 0xffu;
                const unsigned amp = L.N * ((o >> (8 * b)) & 0xffu);
                if (vb < amp) vb = (vb + 1u) & 0xffu; else if (vb > amp) vb = vb - 1u;      // uint8_t ++ wraps
                nv |= vb << (8 * b);
            }
        }
        v[k] = __vmaxu4(__vminu4(nv, vmax4), vmin4);                        // max(min(Vt, Vmax), Vmin) on bytes :581
        ge[k] = __vcmpgeu4(o, v[k]) & 0x01010101u;                          // :604-605
    }
    dps_store12(mp, v12, n, m);
    dps_store12(vp, v12, n, v);
    if (gp) {
        const unsigned p0 = ge[0] & 0x00ffffffu, p1 = __byte_perm(ge[0], ge[1], 0x0543u) & 0x00ffffffu;
        const unsigned p2 = __byte_perm(ge[1], ge[2], 0x0432u) & 0x00ffffffu, p3 = ge[2] >> 8;
        const unsigned mask = (p0 ? 0xffu : 0u) | (p1 ? 0xff00u : 0u) | (p2 ? 0xff0000u : 0u) | (p3 ? 0xff000000u : 0u);
        dps_store_mask(gp, n == 4 && (reinterpret_cast<uintptr_t>(gp) & 3) == 0, n, mask);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Warp-coalesced forms of the two byte-wise models (AdaptiveMedian, SigmaDelta) for launches of whole 512-pixel chunks
// with 16-byte aligned images.  In the 4-pixel kernels above every access is a 32-bit word at a 12-byte stride: three
// instructions walk over the same twelve sectors, and with L1::no_allocate each of them goes to the L2 again -- the kernels
// move three times their bytes between L2 and SM (SigmaDelta: 0.50 of the HBM roofline).  The model arithmetic is
// byte-wise, so it does not care which pixel a byte belongs to: a warp takes 512 pixels = 1536 bytes per image and lane i
// moves bytes [512 k + 16 i, + 16), k = 0..2, with 128-bit accesses (fd_coalesced_kernel's scheme).  Only the mask needs
// whole pixels: the per-byte flags pass through a 1536-byte per-warp shared-memory buffer, from which every lane takes the
// 48 flag bytes of the 16 pixels whose mask bytes it writes.
constexpr int BW_CHUNK_PX = 512, BW_CHUNK_BYTES = BW_CHUNK_PX * 3;

// the 16 mask bytes of a lane from the 1536 flag bytes of its warp (0x01 where a channel says foreground)
__device__ __forceinline__ uint4 bw_mask_from_flags(unsigned char *tbuf, const uint4 (&flags)[3], unsigned lane)
{
    uint4 *tb = reinterpret_cast<uint4 *>(tbuf);
#pragma unroll
    for (int k = 0; k < 3; k++) tb[k * 32 + lane] = flags[k];
    __syncwarp();
    const uint4 *mine = reinterpret_cast<const uint4 *>(tbuf + lane * 48);
    const uint4 a = mine[0], b = mine[1], c = mine[2];
    __syncwarp();
    const unsigned w[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
    unsigned m[4];
#pragma unroll
    for (int g = 0; g < 4; g++) {
        const unsigned w0 = w[3 * g], w1 = w[3 * g + 1], w2 = w[3 * g + 2];
        const unsigned p0 = w0 & 0x00ffffffu, p1 = __byte_perm(w0, w1, 0x0543u) & 0x00ffffffu;
        const unsigned p2 = __byte_perm(w1, w2, 0x0432u) & 0x00ffffffu, p3 = w2 >> 8;
        m[g] = (p0 ? 0xffu : 0u) | (p1 ? 0xff00u : 0u) | (p2 ? 0xff0000u : 0u) | (p3 ? 0xff000000u : 0u);
    }
    return make_uint4(m[0], m[1], m[2], m[3]);
}

__device__ __forceinline__ void bw_ld3(const uint8_t *img, unsigned lane, uint4 (&v)[3])
{
    const uint4 *p = reinterpret_cast<const uint4 *>(img) + lane;
    v[0] = ld_stream_u4(p); v[1] = ld_stream_u4(p + 32); v[2] = ld_stream_u4(p + 64);
}
__device__ __forceinline__ void bw_st3(uint8_t *img, unsigned lane, const uint4 (&v)[3])
{
    uint4 *p = reinterpret_cast<uint4 *>(img) + lane;
    st_stream_u4(p, v[0]); st_stream_u4(p + 32, v[1]); st_stream_u4(p + 64, v[2]);
}

__global__ void __launch_bounds__(256)
sigma_delta_coalesced_kernel(SdLaunch L)
{
    pdl_entry();
    __shared__ __align__(16) unsigned char s_t[8][BW_CHUNK_BYTES];
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const long long chunk = (long long)blockIdx.x * 8 + warp;
    if (chunk >= L.npx / BW_CHUNK_PX) return;                                // whole warps leave
    const size_t s = blockIdx.y, off = (size_t)chunk * BW_CHUNK_BYTES;
    uint8_t *mp = L.Mt + s * L.model_stride + off, *vp = L.Vt + s * L.model_stride + off;
    uint4 in[3], m[3], v[3], ge[3];
    bw_ld3(L.frame + s * L.frame_stride + off, lane, in);
    bw_ld3(mp, lane, m);
    bw_ld3(vp, lane, v);
    const unsigned vmax4 = L.vmax8 * 0x01010101u, vmin4 = L.vmin8 * 0x01010101u;
    auto word = [&](unsigned x, unsigned &mw, unsigned &vw) -> unsigned {     // one word of sigma_delta_kernel's update
        mw = mw + (__vcmpltu4(mw, x) & 0x01010101u) - (__vcmpgtu4(mw, x) & 0x01010101u);
        const unsigned o = __vabs4(__vsub4(mw, x));
        unsigned nv;
        if (L.N == 1u) nv = vw + (__vcmpltu4(vw, o) & 0x01010101u) - (__vcmpgtu4(vw, o) & 0x01010101u);
        else {
            nv = 0u;
#pragma unroll
            for (int b = 0; b < 4; b++) {
                unsigned vb = (vw >> (8 * b)) & 0xffu;
                const unsigned amp = L.N * ((o >> (8 * b)) & 0xffu);
                if (vb < amp) vb = (vb + 1u) & 0xffu; else if (vb > amp) vb = vb - 1u;
                nv |= vb << (8 * b);
            }
        }
        vw = __vmaxu4(__vminu4(nv, vmax4), vmin4);
        return __vcmpgeu4(o, vw) & 0x01010101u;
    };
#pragma unroll
    for (int k = 0; k < 3; k++) {
        ge[k].x = word(in[k].x, m[k].x, v[k].x); ge[k].y = word(in[k].y, m[k].y, v[k].y);
        ge[k].z = word(in[k].z, m[k].z, v[k].z); ge[k].w = word(in[k].w, m[k].w, v[k].w);
    }
    bw_st3(mp, lane, m);
    bw_st3(vp, lane, v);
    const uint4 mask = bw_mask_from_flags(s_t[warp], ge, lane);
    if (L.fg) st_stream_u4(L.fg + s * L.fg_stride + (size_t)chunk * BW_CHUNK_PX + lane * 16u, mask);
}

__global__ void __launch_bounds__(256)
dps_median_coalesced_kernel(DpsLaunch L)
{
    pdl_entry();
    __shared__ __align__(16) unsigned char s_t[8][BW_CHUNK_BYTES];
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const long long chunk = (long long)blockIdx.x * 8 + warp;
    if (chunk >= L.npx / BW_CHUNK_PX) return;
    const size_t s = blockIdx.y, off = (size_t)chunk * BW_CHUNK_BYTES;
    uint8_t *mp = L.median + s * L.median_stride + off;
    uint4 in[3], med[3], gt[3];
    bw_ld3(L.frame + s * L.frame_stride + off, lane, in);
    bw_ld3(mp, lane, med);
    const unsigned hi = L.high_u * 0x01010101u;
    auto flag = [&](unsigned x, unsigned m) { return __vcmpgtu4(__vabsdiffu4(x, m), hi) & 0x01010101u; };
    auto step = [&](unsigned x, unsigned m) { return m + (__vcmpgtu4(x, m) & 0x01010101u) - (__vcmpltu4(x, m) & 0x01010101u); };
#pragma unroll
    for (int k = 0; k < 3; k++) {
        gt[k].x = flag(in[k].x, med[k].x); gt[k].y = flag(in[k].y, med[k].y); gt[k].z = flag(in[k].z, med[k].z); gt[k].w = flag(in[k].w, med[k].w);
    }
    if (L.update) {
#pragma unroll
        for (int k = 0; k < 3; k++) {
            med[k].x = step(in[k].x, med[k].x); med[k].y = step(in[k].y, med[k].y); med[k].z = step(in[k].z, med[k].z); med[k].w = step(in[k].w, med[k].w);
        }
        bw_st3(mp, lane, med);
    }
    const uint4 mask = bw_mask_from_flags(s_t[warp], gt, lane);
    st_stream_u4(L.fg + s * L.fg_stride + (size_t)chunk * BW_CHUNK_PX + lane * 16u, mask);
}

// whole chunks, 16-byte aligned images and strides
static bool bw_coalesced_ok(int npx, int nstreams, std::initializer_list<const void *> ptrs, std::initializer_list<size_t> strides)
{
    if (npx < BW_CHUNK_PX || npx % BW_CHUNK_PX) return false;
    for (const void *p : ptrs) if (reinterpret_cast<uintptr_t>(p) & 15) return false;
    if (nstreams > 1) for (size_t st : strides) if (st & 15) return false;
    return true;
}

int launch_sigma_delta(const SdLaunch &L, int nstreams, cudaStream_t stream)
{
    if (!L.first && bw_coalesced_ok(L.npx, nstreams, {L.frame, L.fg, L.Mt, L.Vt}, {L.frame_stride, L.fg_stride, L.model_stride})) {
        const long long chunks = L.npx / BW_CHUNK_PX;
        launch_pdl(sigma_delta_coalesced_kernel, dim3((unsigned)((chunks + 7) / 8), (unsigned)nstreams), dim3(256), 0, stream, L);
        BGSB_LAUNCH_CHECK();
        return BGSB_OK;
    }
    const long long groups = ((long long)L.npx + 3) / 4;
    launch_pdl(sigma_delta_kernel, dim3((unsigned)((groups + 255) / 256), (unsigned)nstreams), dim3(256), 0, stream, L);
    BGSB_LAUNCH_CHECK();
    return BGSB_OK;
}

int launch_dp_simple(const DpsLaunch &L, int nstreams, cudaStream_t stream)
{
    const long long groups = ((long long)L.npx + 3) / 4;
    const dim3 grid((unsigned)((groups + 255) / 256), (unsigned)nstreams);
    if (L.kind == DPS_MEDIAN && !L.fresh && bw_coalesced_ok(L.npx, nstreams, {L.frame, L.fg, L.median}, {L.frame_stride, L.fg_stride, L.median_stride})) {
        const long long chunks = L.npx / BW_CHUNK_PX;
        launch_pdl(dps_median_coalesced_kernel, dim3((unsigned)((chunks + 7) / 8), (unsigned)nstreams), dim3(256), 0, stream, L);
    } else if (L.kind == DPS_MEDIAN) launch_pdl(dps_median_kernel, grid, dim3(256), 0, stream, L);
    else if (L.kind == DPS_MEAN) launch_pdl(dps_float_kernel<DPS_MEAN>, grid, dim3(256), 0, stream, L);
    else if (L.kind == DPS_WREN) launch_pdl(dps_float_kernel<DPS_WREN>, grid, dim3(256), 0, stream, L);
    else { set_error("launch_dp_simple: bad kind %d", L.kind); return BGSB_ERR_ARG; }
    BGSB_LAUNCH_CHECK();
    return BGSB_OK;
}

}  // namespace bgsb
