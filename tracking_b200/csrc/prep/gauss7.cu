// Pre-processing stage: the reference PreProcessor's gaussianBlur switch, cv::GaussianBlur(img, Size(7, 7), 1.5) on the
// 8-bit BGR frame, as OpenCV 4.x computes it in fixed point (tests/gauss_restate.py restates it in numpy):
//
//     k = (9, 29, 55, 70, 55, 29, 9)                    sum 256
//     out(y, x, c) = (sum_i sum_j k[i] k[j] I(R_h(y + i - 3), R_w(x + j - 3), c) + 2^15) >> 16
//
// R_n is BORDER_REFLECT_101, reflected again as cv::borderInterpolate does when n < 4.  The arithmetic is exact integer,
// so the order of the passes is free: this kernel filters columns first.  A column sum V = sum_i k[i] I is at most
// 65 280 and fits 16 bits, so the column pass carries two bytes per 32-bit word (packed multiply-adds, the symmetric
// taps' rows added first); the row pass of V's stays below 2^24 in 32-bit integers.
//
// Work item = (frame, 16-row group, column strip of STRIP bytes); one 128-thread block each.  Thread t owns the 16-byte
// column chunk [b0 - 16 + 16 t, b0 + 16 t) of the strip, halo chunks included: it keeps the chunk's last 7 input rows in
// registers and slides them down the row group, fetching each row one step ahead, so only 6 of every 22 rows are read
// twice (and those from L2).  Per output row the 128 column sums go to shared memory, and threads 0..125 turn them into
// the 16 output bytes of chunk t + 1 (the halo of 9 bytes each side lies inside the neighbouring chunks).  Interior chunks load and store 128-bit
// words; the frame's first and last 3 pixels, ragged widths and unaligned rows take a per-byte path, and no byte outside
// the frame is read or written.  Output rows [r0, r0 + nr) may be a band of the frame: rows up to 3 beyond the band are
// read, reflected at the frame's edges only.
#include "../common.cuh"
#include "../kernels.h"

namespace bgsb {

namespace {

constexpr int THREADS = 128;
constexpr int STRIP = (THREADS - 2) * 16;       // output bytes of a row per block
constexpr int ROWS = 16;                        // output rows per block
constexpr unsigned K0 = 9, K1 = 29, K2 = 55, K3 = 70;

__device__ __forceinline__ int reflect101(int p, int n)
{
    if (n == 1) return 0;
    while ((unsigned)p >= (unsigned)n) p = p < 0 ? -p : 2 * n - 2 - p;
    return p;
}

// 16 bytes of row `row` at byte offset b (of a row of P bytes); bytes outside [0, P) read as 0 and are never used
__device__ __forceinline__ uint4 fetch_chunk(const uint8_t *row, long long b, int P)
{
    if (b >= 0 && b + 16 <= P && ((uintptr_t)(row + b) & 15) == 0) return *reinterpret_cast<const uint4 *>(row + b);
    unsigned w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int i = 0; i < 16; i++) {
        const long long x = b + i;
        if (x >= 0 && x < P) w[i >> 2] |= (unsigned)row[x] << (8 * (i & 3));
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// the 16 bytes as 8 words of two 16-bit lanes (bytes 2m, 2m + 1)
__device__ __forceinline__ void unpack_chunk(const uint4 v, unsigned (&q)[8])
{
    const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        q[2 * k] = __byte_perm(w[k], 0u, 0x4140);
        q[2 * k + 1] = __byte_perm(w[k], 0u, 0x4342);
    }
}

}  // namespace

__global__ void __launch_bounds__(THREADS) gauss7_kernel(const Gauss7Launch L, long long nitems, int nstrips, int ngroups)
{
    pdl_entry();
    __shared__ __align__(16) unsigned sv[2][THREADS * 8];     // column sums of one output row, two 16-bit lanes per word
    const int t = threadIdx.x;
    const long long item = blockIdx.x;
    if (item >= nitems) return;                               // whole block: the grid has exactly nitems blocks
    const int strip = (int)(item % nstrips);
    const long long rest = item / nstrips;
    const int g = (int)(rest % ngroups);
    const long long f = rest / ngroups;
    const int P = 3 * L.w;
    const int b0 = strip * STRIP;
    const int ya = L.r0 + g * ROWS, nrows = min(ROWS, L.r0 + L.nr - ya);
    const uint8_t *const src = L.src + f * L.frame_stride;
    uint8_t *const dst = L.dst + f * L.frame_stride;
    const long long cb = (long long)b0 - 16 + 16 * t;         // this thread's column chunk

    // the column window: input rows ya - 3 + q in slot q % 7
    unsigned win[7][8];
#pragma unroll
    for (int q = 0; q < 6; q++) unpack_chunk(fetch_chunk(src + (size_t)reflect101(ya - 3 + q, L.h) * P, cb, P), win[q]);
    // the row the next output row adds, fetched one row ahead so its latency overlaps a row's arithmetic and barrier
    uint4 next = fetch_chunk(src + (size_t)reflect101(ya + 3, L.h) * P, cb, P);

    const long long ob = (long long)b0 + 16 * t;              // the output chunk of threads 0..125
    const bool owner = t < THREADS - 2 && ob < P;
    // interior: every tap of the 16 bytes is a byte of the row 3 pixels away at most, without reflection
    const bool interior = ob >= 9 && ob + 16 + 9 <= P;
    for (int m0 = 0; m0 < nrows; m0 += 7) {
#pragma unroll
        for (int u = 0; u < 7; u++) {
            const int m = m0 + u;
            if (m >= nrows) break;                            // uniform over the block
            unpack_chunk(next, win[(u + 6) % 7]);
            if (m + 1 < nrows) next = fetch_chunk(src + (size_t)reflect101(ya + m + 4, L.h) * P, cb, P);
            unsigned *const s = sv[m & 1];
            unsigned v[8];
#pragma unroll
            for (int k = 0; k < 8; k++)
                v[k] = K0 * (win[u % 7][k] + win[(u + 6) % 7][k]) + K1 * (win[(u + 1) % 7][k] + win[(u + 5) % 7][k]) +
                       K2 * (win[(u + 2) % 7][k] + win[(u + 4) % 7][k]) + K3 * win[(u + 3) % 7][k];
            reinterpret_cast<uint4 *>(s)[2 * t] = make_uint4(v[0], v[1], v[2], v[3]);
            reinterpret_cast<uint4 *>(s)[2 * t + 1] = make_uint4(v[4], v[5], v[6], v[7]);
            __syncthreads();                                  // sv[m & 1] was last read for row m - 2, before row m - 1's barrier
            if (owner) {
                uint8_t *const orow = dst + (size_t)(ya + m) * P;
                if (interior) {
                    // column sums of bytes ob - 16 .. ob + 31: words 8t .. 8t + 23 of the row's column sums
                    unsigned cw[24];
#pragma unroll
                    for (int k = 0; k < 6; k++) {
                        const uint4 x = reinterpret_cast<const uint4 *>(s)[2 * t + k];
                        cw[4 * k] = x.x; cw[4 * k + 1] = x.y; cw[4 * k + 2] = x.z; cw[4 * k + 3] = x.w;
                    }
                    unsigned o[4];
#pragma unroll
                    for (int k = 0; k < 4; k++) o[k] = 0;
#pragma unroll
                    for (int j = 0; j < 16; j++) {
#define CS(i) ((cw[(i) >> 1] >> (16 * ((i) & 1))) & 0xffffu)
                        const int c = 16 + j;
                        const unsigned V = 32768u + K3 * CS(c) + K2 * (CS(c - 3) + CS(c + 3)) + K1 * (CS(c - 6) + CS(c + 6)) +
                                           K0 * (CS(c - 9) + CS(c + 9));
#undef CS
                        o[j >> 2] |= (V >> 16) << (8 * (j & 3));
                    }
                    if (ob + 16 <= P && ((uintptr_t)(orow + ob) & 15) == 0) {
                        *reinterpret_cast<uint4 *>(orow + ob) = make_uint4(o[0], o[1], o[2], o[3]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; j++) orow[ob + j] = (uint8_t)(o[j >> 2] >> (8 * (j & 3)));
                    }
                } else {
                    // the frame's first or last 3 pixels, or a ragged chunk: taps reflected at the row's ends; every
                    // reflected tap stays within 9 bytes, inside this strip's halo
                    const unsigned short *const s16 = reinterpret_cast<const unsigned short *>(s);
                    for (int j = 0; j < 16; j++) {
                        const int b = (int)ob + j;
                        if (b >= P) break;
                        const int x = b / 3, ch = b - 3 * x;
                        unsigned V = 32768u;
                        const unsigned kk[7] = {K0, K1, K2, K3, K2, K1, K0};
#pragma unroll
                        for (int d = 0; d < 7; d++) V += kk[d] * s16[3 * reflect101(x + d - 3, L.w) + ch - b0 + 16];
                        orow[b] = (uint8_t)(V >> 16);
                    }
                }
            }
        }
    }
}

int launch_gauss7(const Gauss7Launch &L, cudaStream_t stream)
{
    BGSB_REQUIRE(L.src && L.dst && L.w > 0 && L.h > 0 && L.nframes >= 1, "gauss7: empty frame set");
    BGSB_REQUIRE(L.r0 >= 0 && L.nr >= 1 && L.r0 + L.nr <= L.h, "gauss7: band outside the frame");
    BGSB_REQUIRE((long long)L.w * 3 < (1LL << 31), "gauss7: row too long");
    const int nstrips = (3 * L.w + STRIP - 1) / STRIP, ngroups = (L.nr + ROWS - 1) / ROWS;
    const long long nitems = (long long)L.nframes * ngroups * nstrips;
    BGSB_REQUIRE(nitems < (1LL << 31), "gauss7: frame set too large");
    launch_pdl(gauss7_kernel, dim3((unsigned)nitems), dim3(THREADS), 0, stream, L, nitems, nstrips, ngroups);
    BGSB_LAUNCH_CHECK();
    return BGSB_OK;
}

}  // namespace bgsb
