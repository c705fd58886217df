// K-CCL: 8-connected component labelling of the foreground mask on the GPU, with canonical
// (raster-first) labels, per-component bounding box / area, and the RETR_EXTERNAL nesting test.
//
// Replaces steps 1-2 (and the integer sums of step 4) of CvBlobDetectorCC::DetectNewBlob
// (OpenCV legacy `cvCreateBlobDetectorCC`, referenced at ustc_src/trackingMain.cpp:56,626 and
// readme.md:4-10; spec = SURVEY.md Appendix A.6):
//     cvThreshold(pIB, pIB, 128, 255, CV_THRESH_BINARY); cvFindContours(pIB, ..., CV_RETR_EXTERNAL);
//     CvRect r = ((CvContour*)cnt)->rect;   cvMoments(cvGetSubRect(pFGMask,&mat,r), &m, 0);
//
// Five launches per batch of images (round 1 needed twelve), all one thread per 32-pixel word of the bit-packed
// mask, blockIdx.y = image; no CTA ever waits for another one:
//   1 pack/init  bytes > 128 -> bits (optionally clearing the 1-px frame, OpenCV 2.4 behaviour); every horizontal run
//                inside a word becomes a union-find node named by its first pixel.  (The pipeline's morphology kernel
//                produces the bits and the nodes itself: four launches.)
//   2 merge      unions found with bit tricks on (this row, row above): a run pair is linked exactly once
//                (8-connectivity: vertical + the two diagonals that are not already implied); lock-free union by
//                atomicMin with path halving, so a component's root is its minimum = raster-first pixel.
//   3 roots      every run is pointed straight at its root; a root gets its rank among the roots of its 256-word chunk
//                (kept in its own forest slot as a negative value); the last CTA of an image to finish scans the
//                per-chunk root counts, which makes canonical label = 1 + raster rank of the root a two-load lookup.
//   4 label      labels, bounding boxes / areas by atomics into table rows that need no initialisation (zeroed rows,
//                maxima only); optional label image; the last CTA of an image checks whether any bounding box lies
//                STRICTLY inside another one -- necessary for a component to sit in a hole of another component.
//   5 background one cooperative launch that ends at once unless some image was flagged (typical masks have no such
//                pair: the background is > 98 % of the pixels).  Otherwise the same init / merge / flatten runs on the
//                4-connected background of the flagged images, regions touching the frame are "outer", and a
//                component is external (RETR_EXTERNAL keeps it) iff the background region left of its first pixel is
//                outer.
#include <limits.h>
#include <stdlib.h>
#include <algorithm>
#include <vector>
#include <cooperative_groups.h>

#include "ccl_internal.h"
#include "kernels.h"

namespace cg = cooperative_groups;

namespace bgsb {

constexpr int CCL_TW = 4;                 // width in words of the label kernel's 2-D tiles

__device__ __forceinline__ unsigned in_mask(int k, int w, int wpr)
{
    if (k < 0 || k >= wpr) return 0u;
    if (k < wpr - 1 || (w & 31) == 0) return 0xffffffffu;
    return (1u << (w & 31)) - 1u;
}

// first bit of the run of ones in v that contains bit b
__device__ __forceinline__ int run_start(unsigned v, int b)
{
    unsigned below = ~v & ((b == 0) ? 0u : (0xffffffffu >> (32 - b)));
    return below ? 32 - __clz(below) : 0;
}

__device__ __forceinline__ int find_root(const int *parent, int p)
{
    int q = parent[p];
    while (q != p) { p = q; q = parent[p]; }
    return p;
}

// find with path halving: every visited node is re-pointed at its grandparent.  Re-pointing uses
// atomicMin so that parents only ever decrease (an ancestor always has a smaller index), which keeps
// the lock-free unions below valid while other threads compress the same paths.
__device__ __forceinline__ int find_compress(int *parent, int p)
{
    int q = parent[p];
    while (q != p) {
        int g = parent[q];
        if (g != q) atomicMin(&parent[p], g);
        p = q; q = g;
    }
    return p;
}

__device__ __forceinline__ void unite(int *parent, int a, int b)
{
    while (true) {
        a = find_compress(parent, a);
        b = find_compress(parent, b);
        if (a == b) return;
        if (a < b) { int t = a; a = b; b = t; }      // a > b: hang a under b
        int old = atomicMin(&parent[a], b);
        if (old == a) return;
        a = old;                                      // somebody re-parented a meanwhile: retry
    }
}

// geometry + buffers of one labelling call (all per-image strides are the dense ones of this geometry)
struct CclArgs {
    const unsigned *bits;        // [nimages][h * wpr]
    int *parent;                 // [nimages][w * h]
    uint8_t *outer;              // [nimages][w * h]
    CompRaw *comp;               // [nimages][cap]
    int *chunkcount, *chunkprefix;   // [nimages][nchunks]: roots per 256-word chunk, and their exclusive prefix
    int *done_a, *done_b;        // per image: CTAs of the roots / label kernel that have finished (zero between calls)
    int *ncomp, *need_bg;
    int *labels;                 // [nimages][w * h] or null
    int w, h, wpr, nwords, nchunks, nimages, cap, zero_border, force_bg;
    size_t img_px, img_words;
};

// the (border-cleared) word k of row y; 0 outside the image
__device__ __forceinline__ unsigned ccl_word(const unsigned *bits, int y, int k, const CclArgs &A)
{
    if (k < 0 || k >= A.wpr || y < 0) return 0u;
    return ccl_border(bits[y * A.wpr + k], y, k, A.w, A.h, A.wpr, A.zero_border);
}

// ---- launch 1 (byte masks): pack + node init -------------------------------------------------------------------
__global__ void __launch_bounds__(256)
ccl_pack_kernel(const uint8_t *__restrict__ mask, unsigned *__restrict__ bits, int *__restrict__ parent, int w, int h, int wpr,
                int zero_border, size_t img_px, size_t img_words)
{
    pdl_entry();
    int wi = blockIdx.x * blockDim.x + threadIdx.x;
    if (wi >= h * wpr) return;
    mask += blockIdx.y * img_px; bits += blockIdx.y * img_words; parent += blockIdx.y * img_px;
    int y = wi / wpr, k = wi - y * wpr;
    const uint8_t *p = mask + (size_t)y * w + (size_t)k * 32;
    int nvalid = min(32, w - k * 32);
    unsigned word = 0;
    if (nvalid == 32 && ((reinterpret_cast<uintptr_t>(p) & 15) == 0)) {
        const uint4 *q = reinterpret_cast<const uint4 *>(p);
        uint4 a = __ldg(q), b = __ldg(q + 1);
        unsigned ws[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < 8; i++) {
            unsigned v = ws[i];
            unsigned nz = (((v & 0xffu) > 128u) ? 1u : 0u) | ((((v >> 8) & 0xffu) > 128u) ? 2u : 0u) |
                          ((((v >> 16) & 0xffu) > 128u) ? 4u : 0u) | (((v >> 24) > 128u) ? 8u : 0u);
            word |= nz << (4 * i);
        }
    } else {
        for (int i = 0; i < nvalid; i++) word |= (p[i] > 128 ? 1u : 0u) << i;
    }
    word = ccl_border(word, y, k, w, h, wpr, zero_border);
    bits[wi] = word;
    ccl_init_word(parent, word, y * w + k * 32);
}

template <bool DIAG>
__device__ __forceinline__ void merge_class(int *parent, unsigned v, unsigned vl, unsigned vr, unsigned u,
                                            unsigned ul, unsigned ur, int base, int base_up, bool has_up)
{
    // horizontal continuation across the word boundary
    if ((v & 1u) && (vl >> 31)) unite(parent, base, base - 32 + run_start(vl, 31));
    if (!has_up) return;
    unsigned up_m1 = (u << 1) | (ul >> 31), cur_m1 = (v << 1) | (vl >> 31);
    unsigned A = v & u & ~(cur_m1 & up_m1);
    while (A) {
        int x = __ffs(A) - 1; A &= A - 1;
        unite(parent, base + run_start(v, x), base_up + run_start(u, x));
    }
    if (DIAG) {
        unsigned up_p1 = (u >> 1) | (ur << 31), cur_p1 = (v >> 1) | (vr << 31);
        unsigned B = v & ~u & up_m1 & ~cur_m1;
        while (B) {
            int x = __ffs(B) - 1; B &= B - 1;
            int other = (x == 0) ? base_up - 32 + run_start(ul, 31) : base_up + run_start(u, x - 1);
            unite(parent, base + run_start(v, x), other);
        }
        unsigned C = v & ~u & up_p1 & ~cur_p1;
        while (C) {
            int x = __ffs(C) - 1; C &= C - 1;
            int other = (x == 31) ? base_up + 32 : base_up + run_start(u, x + 1);
            unite(parent, base + run_start(v, x), other);
        }
    }
}

// one word of the merge step.  BG = false: foreground runs, 8-connected;  BG = true: background = complement inside
// the image, 4-connected
template <bool BG>
__device__ __forceinline__ void merge_word(const CclArgs &A, const unsigned *bits, int *parent, int wi)
{
    const int y = wi / A.wpr, k = wi - y * A.wpr;
    const unsigned v = ccl_word(bits, y, k, A);
    if (!BG && v == 0) return;                     // no foreground in this word: nothing to link
    const unsigned vl = ccl_word(bits, y, k - 1, A), vr = ccl_word(bits, y, k + 1, A);
    const bool has_up = y > 0;
    const unsigned u = ccl_word(bits, y - 1, k, A), ul = ccl_word(bits, y - 1, k - 1, A), ur = ccl_word(bits, y - 1, k + 1, A);
    const int base = y * A.w + k * 32, base_up = base - A.w;
    if (!BG) {
        merge_class<true>(parent, v, vl, vr, u, ul, ur, base, base_up, has_up);
    } else {
        const unsigned mk = in_mask(k, A.w, A.wpr), ml = in_mask(k - 1, A.w, A.wpr), mr = in_mask(k + 1, A.w, A.wpr);
        merge_class<false>(parent, ~v & mk, ~vl & ml, ~vr & mr, has_up ? (~u & mk) : 0u, has_up ? (~ul & ml) : 0u,
                           has_up ? (~ur & mr) : 0u, base, base_up, has_up);
    }
}

// Launches 2-4 exist in two shapes: one word per thread (a single image: 254 CTAs at 1080p fill the SMs), and WPT = 4
// words per thread with the loads of the four words in flight together (batches: 16 k CTAs of one word per thread run
// in 14 waves whose CTAs mostly hold empty words and still pay the full launch / arrive latency; a quarter of the
// CTAs does the same work in a quarter of the waves).  A chunk = the 256 * WPT words of one CTA, in raster order:
// word (chunk, j, tid) = chunk * 256 * WPT + j * 256 + tid.

// ---- launch 2: merge ------------------------------------------------------------------------------------------------
template <int WPT>
__global__ void __launch_bounds__(256)
ccl_merge_kernel(const __grid_constant__ CclArgs A)
{
    pdl_entry();
    {   // the table rows the previous call filled go back to zero (the label kernel accumulates into zeroed rows)
        const int nprev = min(A.ncomp[blockIdx.y], A.cap);
        int4 *rows = reinterpret_cast<int4 *>(A.comp + (size_t)blockIdx.y * A.cap);
        for (int i = blockIdx.x * 256 + threadIdx.x; i < 2 * nprev; i += gridDim.x * 256) rows[i] = make_int4(0, 0, 0, 0);
    }
    const unsigned *bits = A.bits + blockIdx.y * A.img_words;
    int *parent = A.parent + blockIdx.y * A.img_px;
    for (int chunk = blockIdx.x; chunk < A.nchunks; chunk += gridDim.x) {
#pragma unroll
        for (int j = 0; j < WPT; j++) {
            const int wi = (chunk * WPT + j) * 256 + threadIdx.x;
            if (wi < A.nwords) merge_word<false>(A, bits, parent, wi);
        }
    }
}

// ---- launch 3: roots ---------------------------------------------------------------------------------------------------
// Every run finds its root (merge has completed: a root is a node that is its own parent) and points straight at it; a
// root gets its rank AMONG THE ROOTS OF ITS CHUNK, stored in its own forest slot as ~rank (< 0); the chunk's root count
// goes to chunkcount[].  The last CTA of an image to finish turns the counts into exclusive prefixes (chunkprefix[]) and
// the component count -- no CTA ever waits for another.
template <int WPT>
__global__ void __launch_bounds__(256)
ccl_roots_kernel(const __grid_constant__ CclArgs A)
{
    pdl_entry();
    __shared__ int wsum[8];
    __shared__ int s_last, s_carry;
    const int img = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const unsigned *bits = A.bits + img * A.img_words;
    int *parent = A.parent + img * A.img_px;
    int *count = A.chunkcount + (size_t)img * A.nchunks;
    // one chunk per CTA, or (capped grids: the pipeline beside the plugin kernel) the CTA's share of the image's chunks
    for (int chunk = blockIdx.x; chunk < A.nchunks; chunk += gridDim.x) {
    unsigned v[WPT], roots[WPT];
    int base[WPT];
#pragma unroll
    for (int j = 0; j < WPT; j++) {
        const int wi = (chunk * WPT + j) * 256 + tid;
        const bool valid = wi < A.nwords;
        const int y = valid ? wi / A.wpr : 0, k = valid ? wi - y * A.wpr : 0;
        v[j] = valid ? ccl_word(bits, y, k, A) : 0u;
        base[j] = y * A.w + k * 32;
    }
    {   // most chunks of a typical mask hold no foreground at all: nothing to rank
        unsigned any = 0;
#pragma unroll
        for (int j = 0; j < WPT; j++) any |= v[j];
        if (!__syncthreads_or(any != 0u)) {
            if (tid == 0) count[chunk] = 0;
            continue;
        }
    }
#pragma unroll
    for (int j = 0; j < WPT; j++) {
        roots[j] = 0;
        for (unsigned s = v[j] & ~(v[j] << 1); s;) {
            const int b = __ffs(s) - 1; s &= s - 1;
            const int p = base[j] + b;
            int cur = p, q = parent[cur];
            while (q != cur && q >= 0) { cur = q; q = parent[cur]; }     // q < 0: that root already carries its rank
            if (cur == p) roots[j] |= 1u << b;
            else parent[p] = cur;
        }
    }
    int carry = 0;                                   // roots of this chunk in the word groups before j
#pragma unroll
    for (int j = 0; j < WPT; j++) {
        const int c = __popc(roots[j]);
        int incl = c;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= off) incl += t;
        }
        if (j) __syncthreads();                      // wsum of the previous group has been read
        if (lane == 31) wsum[wid] = incl;
        __syncthreads();
        int before = 0, total = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) { const int t = wsum[i]; if (i < wid) before += t; total += t; }
        int run = carry + before + incl - c;
        for (unsigned r = roots[j]; r;) {
            const int b = __ffs(r) - 1; r &= r - 1;
            parent[base[j] + b] = ~run;
            run++;
        }
        carry += total;
    }
    if (tid == 0) count[chunk] = carry;
    __syncthreads();                                   // wsum is reused by the CTA's next chunk
    }
    // the last CTA of the image: exclusive scan of the chunk counts.  (One fence by the arriving thread is enough: the
    // barrier orders the CTA's writes before it, and fences are cumulative.)
    __syncthreads();
    if (tid == 0) { __threadfence(); s_last = (atomicAdd(&A.done_a[img], 1) == (int)gridDim.x - 1); s_carry = 0; }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    int *prefix = A.chunkprefix + (size_t)img * A.nchunks;
    for (int c0 = 0; c0 < A.nchunks; c0 += 256) {
        const int j = c0 + tid;
        const int cnt = j < A.nchunks ? __ldcg(count + j) : 0;
        int inc2 = cnt;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc2, off);
            if (lane >= off) inc2 += t;
        }
        __syncthreads();                               // wsum / s_carry of the previous round have been read
        if (lane == 31) wsum[wid] = inc2;
        __syncthreads();
        int bef = s_carry, tot = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) { const int t = wsum[i]; if (i < wid) bef += t; tot += t; }
        if (j < A.nchunks) prefix[j] = bef + inc2 - cnt;
        __syncthreads();
        if (tid == 0) s_carry += tot;
    }
    __syncthreads();
    if (tid == 0) A.ncomp[img] = s_carry;
}

// canonical label = 1 + (roots in the chunks before the root's chunk) + (the root's rank inside its chunk).  The table
// rows are zero on entry and are only ever touched by atomics (and by the root's own thread for the fields nobody else
// writes), so no row has to be initialised before another CTA may use it: maxima as they are, minima as CCL_BIG - value.
constexpr int CCL_BIG = 1 << 30;

// The last CTA of an image decides whether the image needs the background pass: does any component's bounding box lie
// strictly inside another's?  (Necessary for a component to sit in a hole of another one.)  More than 1024 components:
// not worth checking in one CTA, take the pass.
__device__ __forceinline__ void ccl_nest_check(const CclArgs &A, int img, const CompRaw *comp, int4 *s_box, int tid)
{
    const int n = __ldcg(A.ncomp + img);
    int need = 0;
    if (A.force_bg || n > 1024 || n > A.cap) need = (n > 0) || A.force_bg;
    else {
        int4 mine[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int i = u * 256 + tid;
            mine[u] = make_int4(0, 0, 0, 0);
            if (i < n) mine[u] = make_int4(CCL_BIG - __ldcg(&comp[i].xmin), CCL_BIG - __ldcg(&comp[i].ymin), __ldcg(&comp[i].xmax), __ldcg(&comp[i].ymax));
        }
#pragma unroll
        for (int tt = 0; tt < 4; tt++) {
            if (tt * 256 < n) {                        // uniform over the CTA
                s_box[tid] = (tt * 256 + tid < n) ? mine[tt] : make_int4(1 << 30, 1 << 30, -1, -1);
                __syncthreads();
                const int m = min(256, n - tt * 256);
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    if (u * 256 + tid < n) {
                        for (int q2 = 0; q2 < m; q2++) {
                            const int4 bx = s_box[q2];
                            need |= (bx.x < mine[u].x) & (bx.y < mine[u].y) & (bx.z > mine[u].z) & (bx.w > mine[u].w);
                        }
                    }
                }
                __syncthreads();
            }
        }
    }
    need = __syncthreads_or(need);
    if (tid == 0) {
        A.need_bg[img] = need ? 1 : 0;               // every image of the call gets its answer (no stale flags)
        A.done_a[img] = 0; A.done_b[img] = 0;        // both kernels' CTAs have all arrived: zero again for the next call
    }
}

// ---- launch 4: label ------------------------------------------------------------------------------------------------
// A CTA owns a 2-D tile of 4 words x 64 * WPT rows, so that a component's statistics leave the CTA ONCE: a blob of the
// size the tracker cares about lies in a handful of such tiles (a raster chunk of 256 words is 4 rows of a 1080p mask).
// The runs of the tile accumulate bounding box and area in a small shared-memory table keyed by the root; one thread
// per occupied slot looks the component's rank up and issues the five global atomics; with LABELS the runs then read
// the rank back from the table.  (The first round-2 kernel worked on raster chunks and sent five atomics PER RUN to the
// component's row -- 1600 same-sector atomics for a 100 x 80 blob: 15 us on a single 1080p mask; this form: one mask
// 35 -> 29 us, 64 masks 200 -> 154 us.)  Tiles of noise (many runs per word, more components than slots) and runs that
// find no slot take the per-run path.
constexpr int CCL_NS = 128;               // slots of the per-CTA table
constexpr int CCL_PROBES = 8;

template <int WPT>
__device__ __forceinline__ int ccl_rank_of_root(const CclArgs &A, const int *parent, const int *prefix, int root, int local)
{
    constexpr int CSHIFT = WPT == 1 ? 8 : 10;
    const int ry = root / A.w, rx = root - ry * A.w;
    return prefix[(ry * A.wpr + (rx >> 5)) >> CSHIFT] + local;
}

template <bool LABELS, int WPT>
__global__ void __launch_bounds__(256)
ccl_label_tile_kernel(const __grid_constant__ CclArgs A)
{
    pdl_entry();
    __shared__ int4 s_box[256];
    __shared__ int4 s_stage[LABELS ? 8 * 256 : 1];
    __shared__ int s_key[CCL_NS], s_val[CCL_NS][5], s_rank[CCL_NS];
    __shared__ int s_last;
    static_assert(WPT == 1 || WPT == 4, "chunk sizes 256 / 1024 words");
    const int img = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned *bits = A.bits + img * A.img_words;
    const int *parent = A.parent + img * A.img_px;
    const int *prefix = A.chunkprefix + (size_t)img * A.nchunks;
    CompRaw *comp = A.comp + (size_t)img * A.cap;
    constexpr int TH = 64 * WPT;
    const int ntx = (A.wpr + CCL_TW - 1) / CCL_TW, nty = (A.h + TH - 1) / TH, ntiles = ntx * nty;
    const int col = tid & 3, row = tid >> 2;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int ty = tile / ntx, tx = tile - ty * ntx;
        const int k = tx * CCL_TW + col;
        for (int i = tid; i < CCL_NS; i += 256) {
            s_key[i] = -1; s_val[i][0] = 0; s_val[i][1] = 0; s_val[i][2] = 0; s_val[i][3] = 0; s_val[i][4] = 0;
        }
        unsigned v[WPT];
        int yy[WPT];
        unsigned any = 0;
#pragma unroll
        for (int j = 0; j < WPT; j++) {
            const int y = ty * TH + j * 64 + row;
            const bool valid = k < A.wpr && y < A.h;
            yy[j] = valid ? y : -1;
            v[j] = valid ? ccl_word(bits, y, k, A) : 0u;
            any |= v[j];
        }
        const bool work = __syncthreads_or(any != 0u);           // also: the table is initialised
        // a tile of noise (many runs per word) holds more components than the table has slots: per-run path at once
        bool dense = false;
        if (work) {
            int heavy = 0;
#pragma unroll
            for (int j = 0; j < WPT; j++) heavy |= __popc(v[j] & ~(v[j] << 1)) >= 3;
            dense = __syncthreads_count(heavy) > 32;
        }
        const int probes = dense ? 0 : CCL_PROBES;
        if (work) {
            // phase 1: every run adds itself to its root's slot
#pragma unroll
            for (int j = 0; j < WPT; j++) {
                const int y = yy[j];
                const int base = y * A.w + k * 32;
                for (unsigned s = v[j] & ~(v[j] << 1); s;) {
                    const int b = __ffs(s) - 1; s &= s - 1;
                    const int p = base + b;
                    const int q = parent[p];
                    const int root = q < 0 ? p : q;
                    const unsigned rest = ~(v[j] >> b);
                    const int len = rest ? __ffs(rest) - 1 : 32 - b;
                    const int x0 = k * 32 + b;
                    if (q < 0) {                                    // the root's own thread: fields nobody else writes
                        const int rank = ccl_rank_of_root<WPT>(A, parent, prefix, p, ~q);
                        if (rank < A.cap) { CompRaw *cp = comp + rank; cp->label = rank + 1; cp->first_index = p; cp->external = 1; }
                    }
                    unsigned hsh = ((unsigned)root * 2654435761u) >> 25;      // 7 bits
                    bool placed = false;
#pragma unroll 1
                    for (int t = 0; t < probes && !placed; t++) {
                        const int old = atomicCAS(&s_key[hsh], -1, root);
                        if (old == -1 || old == root) {
                            atomicMax(&s_val[hsh][0], CCL_BIG - x0); atomicMax(&s_val[hsh][1], x0 + len - 1);
                            atomicMax(&s_val[hsh][2], CCL_BIG - y); atomicMax(&s_val[hsh][3], y);
                            atomicAdd(&s_val[hsh][4], len);
                            placed = true;
                        } else hsh = (hsh + 1) & (CCL_NS - 1);
                    }
                    if (!placed) {                                  // crowded tile: this run goes to the row itself
                        const int rank = ccl_rank_of_root<WPT>(A, parent, prefix, root, ~(q < 0 ? q : parent[root]));
                        if (rank < A.cap) {
                            CompRaw *cp = comp + rank;
                            atomicMax(&cp->xmin, CCL_BIG - x0); atomicMax(&cp->xmax, x0 + len - 1);
                            atomicMax(&cp->ymin, CCL_BIG - y); atomicMax(&cp->ymax, y);
                            atomicAdd(&cp->area, len);
                        }
                    }
                }
            }
            __syncthreads();
            // phase 2: one thread per occupied slot: rank of the component, its statistics to the table row
            if (tid < CCL_NS && s_key[tid] >= 0) {
                const int root = s_key[tid];
                const int rank = ccl_rank_of_root<WPT>(A, parent, prefix, root, ~parent[root]);
                s_rank[tid] = rank;
                if (rank < A.cap) {
                    CompRaw *cp = comp + rank;
                    atomicMax(&cp->xmin, s_val[tid][0]); atomicMax(&cp->xmax, s_val[tid][1]);
                    atomicMax(&cp->ymin, s_val[tid][2]); atomicMax(&cp->ymax, s_val[tid][3]);
                    atomicAdd(&cp->area, s_val[tid][4]);
                }
            }
        }
        if (LABELS) {
            if (work) __syncthreads();                              // s_rank is complete
#pragma unroll
            for (int j = 0; j < WPT; j++) {
                const int y = yy[j];
                const int base = y * A.w + k * 32;
                int lab[32];
#pragma unroll
                for (int i = 0; i < 32; i++) lab[i] = 0;
                for (unsigned s = v[j] & ~(v[j] << 1); s;) {
                    const int b = __ffs(s) - 1; s &= s - 1;
                    const int p = base + b;
                    const int q = parent[p];
                    const int root = q < 0 ? p : q;
                    unsigned hsh = ((unsigned)root * 2654435761u) >> 25;
                    int rank = -1;
#pragma unroll 1
                    for (int t = 0; t < probes && rank < 0; t++) {
                        const int key = s_key[hsh];
                        if (key == root) rank = s_rank[hsh];
                        else if (key == -1) break;
                        else hsh = (hsh + 1) & (CCL_NS - 1);
                    }
                    if (rank < 0) rank = ccl_rank_of_root<WPT>(A, parent, prefix, root, ~(q < 0 ? q : parent[root]));
                    const unsigned rest = ~(v[j] >> b);
                    const int len = rest ? __ffs(rest) - 1 : 32 - b;
#pragma unroll
                    for (int i = 0; i < 32; i++)
                        if (i >= b && i < b + len) lab[i] = rank + 1;
                }
                // the warp's 32 words are 8 rows x 4 words: per row 512 contiguous bytes of the label image
                int *limg = A.labels + img * A.img_px;
                const int y0 = ty * TH + j * 64 + warp * 8;          // the warp's first row
                const bool whole = (A.w & 31) == 0 && tx * CCL_TW + CCL_TW <= A.wpr &&
                                   (reinterpret_cast<uintptr_t>(limg + (size_t)y0 * A.w + tx * CCL_TW * 32) & 15) == 0;
                if (whole) {
                    const bool empty = __ballot_sync(0xffffffffu, v[j] != 0u) == 0u;
                    int4 *stage = s_stage + warp * 256;
                    if (!empty) {
#pragma unroll
                        for (int i = 0; i < 8; i++)
                            stage[lane * 8 + (i ^ (lane & 7))] = make_int4(lab[4 * i], lab[4 * i + 1], lab[4 * i + 2], lab[4 * i + 3]);
                        __syncwarp();
                    }
#pragma unroll
                    for (int q = 0; q < 8; q++) {
                        if (y0 + q < A.h) {
                            const int sw = q * 4 + (lane >> 3), part = lane & 7;       // source thread of the warp, its int4
                            int4 *dst = reinterpret_cast<int4 *>(limg + (size_t)(y0 + q) * A.w + tx * CCL_TW * 32) + lane;
                            *dst = empty ? make_int4(0, 0, 0, 0) : stage[sw * 8 + (part ^ (sw & 7))];
                        }
                    }
                    __syncwarp();
                } else if (y >= 0) {
                    int *o = limg + base;
                    const int nvalid = min(32, A.w - k * 32);
                    if (nvalid == 32 && ((reinterpret_cast<uintptr_t>(o) & 15) == 0)) {
#pragma unroll
                        for (int i = 0; i < 8; i++)
                            reinterpret_cast<int4 *>(o)[i] = make_int4(lab[4 * i], lab[4 * i + 1], lab[4 * i + 2], lab[4 * i + 3]);
                    } else {
#pragma unroll
                        for (int i = 0; i < 32; i++)
                            if (i < nvalid) o[i] = lab[i];
                    }
                }
            }
        }
        __syncthreads();                                            // the table is reused by the CTA's next tile
    }
    // ---- the last CTA of the image: does the image need the background pass?
    __syncthreads();
    if (tid == 0) { __threadfence(); s_last = (atomicAdd(&A.done_b[img], 1) == (int)gridDim.x - 1); }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    ccl_nest_check(A, img, comp, s_box, tid);
}

// ---- launch 5: RETR_EXTERNAL ------------------------------------------------------------------------------------------
// the background pass, one word / one component at a time
__device__ __forceinline__ void bg_init_word(const CclArgs &A, int img, int wi)
{
    const unsigned *bits = A.bits + img * A.img_words;
    int *parent = A.parent + img * A.img_px;
    uint8_t *outer = A.outer + img * A.img_px;
    const int y = wi / A.wpr, k = wi - y * A.wpr;
    const unsigned vb = ~ccl_word(bits, y, k, A) & in_mask(k, A.w, A.wpr);
    const int base = y * A.w + k * 32;
    for (unsigned s = vb & ~(vb << 1); s;) {
        const int b = __ffs(s) - 1; s &= s - 1;
        parent[base + b] = base + b;
        outer[base + b] = 0;
    }
}
// flatten; regions that touch the image frame are "outer"
__device__ __forceinline__ void bg_flatten_word(const CclArgs &A, int img, int wi)
{
    const unsigned *bits = A.bits + img * A.img_words;
    int *parent = A.parent + img * A.img_px;
    uint8_t *outer = A.outer + img * A.img_px;
    const int y = wi / A.wpr, k = wi - y * A.wpr;
    const unsigned vb = ~ccl_word(bits, y, k, A) & in_mask(k, A.w, A.wpr);
    const int base = y * A.w + k * 32;
    const bool edge_row = (y == 0 || y == A.h - 1);
    for (unsigned s = vb & ~(vb << 1); s;) {
        const int b = __ffs(s) - 1; s &= s - 1;
        const int r = find_root(parent, base + b);
        parent[base + b] = r;
        const unsigned rest = ~(vb >> b);
        const int len = rest ? __ffs(rest) - 1 : 32 - b;
        if (edge_row || (k == 0 && b == 0) || (k * 32 + b + len - 1 == A.w - 1)) outer[r] = 1;
    }
}
// a component is external iff the background region left of its first pixel is outer
__device__ __forceinline__ void bg_resolve_comp(const CclArgs &A, int img, int i)
{
    const unsigned *bits = A.bits + img * A.img_words;
    const int *parent = A.parent + img * A.img_px;
    const uint8_t *outer = A.outer + img * A.img_px;
    CompRaw *c = A.comp + (size_t)img * A.cap + i;
    const int r = c->first_index;
    const int ry = r / A.w, rx = r - ry * A.w;
    int ext = 1;
    if (rx > 0) {
        const int lk = (rx - 1) >> 5, lb = (rx - 1) & 31;
        const unsigned lv = ~ccl_word(bits, ry, lk, A) & in_mask(lk, A.w, A.wpr);
        ext = outer[parent[ry * A.w + lk * 32 + run_start(lv, lb)]];
    }
    c->external = ext;
}

// One cooperative launch (grid-wide barriers between the phases): the form for a labeller that has the GPU to itself.
__global__ void __launch_bounds__(256)
ccl_background_kernel(const __grid_constant__ CclArgs A)
{
    pdl_entry();
    cg::grid_group grid = cg::this_grid();
    const int tid = threadIdx.x;
    const size_t gtid = (size_t)blockIdx.x * 256 + tid, gsize = (size_t)gridDim.x * 256;
    // the label kernel's last CTA per image has flagged the images where a bounding box lies strictly inside another
    int any = 0;
    for (int i = tid; i < A.nimages; i += 256) any |= A.need_bg[i];
    if (!__syncthreads_or(any)) return;              // the same answer in every CTA: typical masks end here

    // The phases stride over (image, word) pairs of ALL images at once: the background of an image is essentially one
    // huge component, whose unions contend on one root -- latency, not throughput -- so flagged images must progress
    // side by side, not one after the other.
    const size_t nitems = (size_t)A.nimages * A.nwords;
    for (size_t it = gtid; it < nitems; it += gsize) {
        const int img = (int)(it / A.nwords), wi = (int)(it - (size_t)img * A.nwords);
        if (A.need_bg[img]) bg_init_word(A, img, wi);
    }
    grid.sync();
    for (size_t it = gtid; it < nitems; it += gsize) {
        const int img = (int)(it / A.nwords), wi = (int)(it - (size_t)img * A.nwords);
        if (A.need_bg[img]) merge_word<true>(A, A.bits + img * A.img_words, A.parent + img * A.img_px, wi);
    }
    grid.sync();
    for (size_t it = gtid; it < nitems; it += gsize) {
        const int img = (int)(it / A.nwords), wi = (int)(it - (size_t)img * A.nwords);
        if (A.need_bg[img]) bg_flatten_word(A, img, wi);
    }
    grid.sync();
    for (int img = 0; img < A.nimages; img++) {
        if (!A.need_bg[img]) continue;
        const int n = min(A.ncomp[img], A.cap);
        for (size_t i = gtid; i < (size_t)n; i += gsize) bg_resolve_comp(A, img, (int)i);
    }
}

// The same pass as four plain launches (PHASE 0 init, 1 merge, 2 flatten, 3 resolve), grid (X, images), whose CTAs leave at
// once for images that were not flagged: the form for the pipeline, where the labeller runs BESIDE the next frame
// set's plugin kernel -- a cooperative grid would have to wait until that kernel has drained to become resident as a
// whole, and the plugin kernel after it would wait for the labeller.
template <int PHASE>
__global__ void __launch_bounds__(256)
ccl_background_phase_kernel(const __grid_constant__ CclArgs A)
{
    pdl_entry();
    const int img = blockIdx.y;
    if (!A.need_bg[img]) return;
    const int limit = PHASE == 3 ? min(A.ncomp[img], A.cap) : A.nwords;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < limit; i += gridDim.x * 256) {
        if (PHASE == 0) bg_init_word(A, img, i);
        else if (PHASE == 1) merge_word<true>(A, A.bits + img * A.img_words, A.parent + img * A.img_px, i);
        else if (PHASE == 2) bg_flatten_word(A, img, i);
        else bg_resolve_comp(A, img, i);
    }
}

// cvMoments(ROI, binary=0): pixel-value weighted raw moments, ROI-relative coordinates.
__global__ void __launch_bounds__(256)
rect_moments_kernel(const uint8_t *__restrict__ mask, int w, int h, const int *__restrict__ rects,
                    unsigned long long *out)
{
    pdl_entry();
    const int ri = blockIdx.x;
    const int rx = rects[4 * ri], ry = rects[4 * ri + 1], rw = rects[4 * ri + 2], rh = rects[4 * ri + 3];
    unsigned long long m[6] = {0, 0, 0, 0, 0, 0};
    // each y-slice of blocks takes every gridDim.y-th row
    for (int yy = blockIdx.y; yy < rh; yy += gridDim.y) {
        int y = ry + yy;
        if (y < 0 || y >= h) continue;
        const uint8_t *row = mask + (size_t)y * w;
        unsigned long long r0 = 0, r1 = 0, r2 = 0;       // sum v, sum v*x, sum v*x*x over this row
        for (int xx = threadIdx.x; xx < rw; xx += blockDim.x) {
            int x = rx + xx;
            if (x < 0 || x >= w) continue;
            unsigned long long v = row[x];
            r0 += v; r1 += v * xx; r2 += v * (unsigned long long)xx * xx;
        }
        m[0] += r0; m[1] += r1; m[2] += r0 * yy; m[3] += r2; m[4] += r0 * (unsigned long long)yy * yy; m[5] += r1 * yy;
    }
    __shared__ unsigned long long red[6][8];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 6; i++) {
        unsigned long long v = m[i];
        for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
        if (lane == 0) red[i][wid] = v;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        unsigned long long v = 0;
        for (int i = 0; i < 8; i++) v += red[threadIdx.x][i];
        if (v) atomicAdd(out + 6 * ri + threadIdx.x, v);
    }
}

// The same sums from a bit-packed {0,255} mask (the pipeline keeps no byte mask): every set bit weighs 255.
__global__ void __launch_bounds__(256)
rect_moments_bits_kernel(const unsigned *__restrict__ bits, int w, int h, int wpr, const int *__restrict__ rects,
                         unsigned long long *out)
{
    pdl_entry();
    const int ri = blockIdx.x;
    const int rx = rects[4 * ri], ry = rects[4 * ri + 1], rw = rects[4 * ri + 2], rh = rects[4 * ri + 3];
    const int xa = max(rx, 0), xb = min(rx + rw, w);             // [xa, xb) inside the image
    unsigned long long m[6] = {0, 0, 0, 0, 0, 0};
    if (xa < xb) {
        const int k0 = xa >> 5, k1 = (xb - 1) >> 5;
        for (int yy = blockIdx.y; yy < rh; yy += gridDim.y) {
            const int y = ry + yy;
            if (y < 0 || y >= h) continue;
            unsigned long long r0 = 0, r1 = 0, r2 = 0;
            for (int k = k0 + (int)threadIdx.x; k <= k1; k += blockDim.x) {
                unsigned v = bits[(size_t)y * wpr + k];
                if (k == k0) v &= 0xffffffffu << (xa & 31);
                if (k == k1 && (xb & 31)) v &= 0xffffffffu >> (32 - (xb & 31));
                while (v) {
                    const int b = __ffs(v) - 1; v &= v - 1;
                    const unsigned long long xx = (unsigned long long)(k * 32 + b - rx);
                    r0 += 255ull; r1 += 255ull * xx; r2 += 255ull * xx * xx;
                }
            }
            m[0] += r0; m[1] += r1; m[2] += r0 * yy; m[3] += r2; m[4] += r0 * (unsigned long long)yy * yy; m[5] += r1 * yy;
        }
    }
    __shared__ unsigned long long red[6][8];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 6; i++) {
        unsigned long long v = m[i];
        for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
        if (lane == 0) red[i][wid] = v;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        unsigned long long v = 0;
        for (int i = 0; i < 8; i++) v += red[threadIdx.x][i];
        if (v) atomicAdd(out + 6 * ri + threadIdx.x, v);
    }
}

// The component tables of all images of the last call, decoded, in one dense buffer: per image 8 ints of header
// (count, 7 x 0) followed by `rows` bgsb_component rows (x, y, w, h form); one download then serves a whole stream group.
__global__ void __launch_bounds__(256)
ccl_gather_kernel(const CompRaw *__restrict__ comp, const int *__restrict__ ncomp, int cap, int rows, int *__restrict__ out)
{
    pdl_entry();
    const int img = blockIdx.x;
    const int n = ncomp[img];
    int *o = out + (size_t)img * (rows + 1) * 8;
    if (threadIdx.x < 8) o[threadIdx.x] = threadIdx.x == 0 ? n : 0;
    const int m = min(min(n, rows), cap);
    const CompRaw *c = comp + (size_t)img * cap;
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
        const CompRaw r = c[i];
        const int x = CCL_BIG - r.xmin, y = CCL_BIG - r.ymin;
        int4 *d = reinterpret_cast<int4 *>(o + (size_t)(i + 1) * 8);
        d[0] = make_int4(r.label, r.first_index, x, y);
        d[1] = make_int4(r.xmax - x + 1, r.ymax - y + 1, r.area, r.external);
    }
}

int ccl_gather_tables(bgsb_ccl *c, int32_t *d_out, int rows, cudaStream_t stream)
{
    BGSB_REQUIRE(c && d_out && rows >= 0, "bad args");
    if (!c->labelled) { set_error("ccl_gather_tables: nothing labelled yet"); return BGSB_ERR_STATE; }
    launch_pdl(ccl_gather_kernel, dim3(c->nimages), dim3(256), 0, stream, (const CompRaw *)c->d_comp, (const int *)c->d_ncomp, c->cap,
               rows, (int *)d_out);
    BGSB_LAUNCH_CHECK();
    return BGSB_OK;
}

// launches 2-4 (the producer of the words has created the nodes)
int ccl_label_bits(bgsb_ccl *c, const unsigned *d_bits, int w, int h, int nimages, int zero_border,
                   int32_t *d_labels, cudaStream_t stream)
{
    BGSB_REQUIRE(c && d_bits, "null");
    BGSB_REQUIRE(w > 0 && h > 0 && w <= c->max_w && h <= c->max_h, "image larger than the labeller was created for");
    BGSB_REQUIRE(nimages >= 1 && nimages <= c->max_images, "more images than the labeller was created for");
    BGSB_CUDA(cudaSetDevice(c->device));
    CclArgs A;
    memset(&A, 0, sizeof(A));
    A.bits = d_bits; A.parent = c->d_parent; A.outer = c->d_outer; A.comp = c->d_comp;
    A.chunkcount = c->d_chunkcount; A.chunkprefix = c->d_chunkprefix; A.done_a = c->d_done; A.done_b = c->d_done + c->max_images;
    A.ncomp = c->d_ncomp; A.need_bg = c->d_need_bg; A.labels = d_labels;
    A.w = w; A.h = h; A.wpr = (w + 31) / 32; A.nwords = A.wpr * h; A.nchunks = (A.nwords + 255) / 256;
    A.nimages = nimages; A.cap = c->cap; A.zero_border = zero_border; A.force_bg = c->force_bg;

    A.img_px = (size_t)w * h; A.img_words = (size_t)A.nwords;      // dense per-image strides for this geometry
    if (c->dirty) {                                 // an earlier call failed between the launches
        BGSB_CUDA(cudaMemsetAsync(c->d_done, 0, 2 * (size_t)c->max_images * sizeof(int), stream));
        BGSB_CUDA(cudaMemsetAsync(c->d_need_bg, 0, (size_t)c->max_images * sizeof(int), stream));
    }
    if (nimages < c->table_images) {
        // fewer images than the previous call: the rows of the images that now sit out are cleared here (the merge kernel
        // clears those of the images it works on)
        const size_t first = (size_t)nimages, cnt = (size_t)(c->table_images - nimages);
        BGSB_CUDA(cudaMemsetAsync(c->d_comp + first * c->cap, 0, cnt * c->cap * sizeof(CompRaw), stream));
        BGSB_CUDA(cudaMemsetAsync(c->d_ncomp + first, 0, cnt * sizeof(int), stream));
    }
    c->table_images = nimages;
    c->dirty = true;
    const dim3 block(256);
    // Words per thread: 1 for a single image (254 CTAs at 1080p fill the SMs), 4 for batches too big for one wave of
    // one-word CTAs.  (16 words per thread was measured and removed: a sixteenth of the CTAs, but the per-word work of a
    // thread is serial -- 64 masks 166 -> 284 us, 8 masks 44 -> 117 us.)
    const long long n256 = (long long)nimages * ((A.nwords + 255) / 256);
    const int wpt = n256 > 8LL * sm_count(c->device) ? 4 : 1;
    A.nchunks = (A.nwords + 256 * wpt - 1) / (256 * wpt);
    // (the kernels loop over chunks, so capped grids work; measured, capping them beside the plugin kernel only makes
    // the chain longer: tools/chain_ctas_probe.py)
    const dim3 grid(A.nchunks, nimages);
#define BGSB_CCL_LAUNCH(W)                                                                                      \
    do {                                                                                                        \
        launch_pdl(ccl_merge_kernel<W>, grid, block, 0, stream, A);                                             \
        BGSB_LAUNCH_CHECK();                                                                                    \
        launch_pdl(ccl_roots_kernel<W>, grid, block, 0, stream, A);                                             \
        BGSB_LAUNCH_CHECK();                                                                                    \
        const dim3 tgrid(((A.wpr + CCL_TW - 1) / CCL_TW) * ((A.h + 64 * W - 1) / (64 * W)), nimages);           \
        if (d_labels) launch_pdl(ccl_label_tile_kernel<true, W>, tgrid, block, 0, stream, A);                   \
        else launch_pdl(ccl_label_tile_kernel<false, W>, tgrid, block, 0, stream, A);                           \
        BGSB_LAUNCH_CHECK();                                                                                    \
    } while (0)
    if (wpt == 4) BGSB_CCL_LAUNCH(4);
    else BGSB_CCL_LAUNCH(1);
#undef BGSB_CCL_LAUNCH
    if (c->max_ctas > 0) {
        // beside another kernel (pipeline): four plain launches that leave at once for images that were not flagged
        const dim3 bgrid(std::max(1, std::min((A.nwords + 255) / 256, c->max_ctas / nimages)), nimages);
        launch_pdl(ccl_background_phase_kernel<0>, bgrid, block, 0, stream, A);
        BGSB_LAUNCH_CHECK();
        launch_pdl(ccl_background_phase_kernel<1>, bgrid, block, 0, stream, A);
        BGSB_LAUNCH_CHECK();
        launch_pdl(ccl_background_phase_kernel<2>, bgrid, block, 0, stream, A);
        BGSB_LAUNCH_CHECK();
        launch_pdl(ccl_background_phase_kernel<3>, bgrid, block, 0, stream, A);
        BGSB_LAUNCH_CHECK();
    } else {
        // cooperative: every CTA must be resident at once; the grid strides over the work
        if (c->coop_ctas <= 0) {
            int per_sm = 0;
            BGSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ccl_background_kernel, 256, 0));
            c->coop_ctas = std::min(4, std::max(1, per_sm)) * sm_count(c->device);
        }
        const long long want = (long long)nimages * ((A.nwords + 255) / 256);
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)std::min<long long>(c->coop_ctas, std::max<long long>(want, 1)));
        cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeCooperative;
        attr[0].val.cooperative = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        const cudaError_t e = cudaLaunchKernelEx(&cfg, ccl_background_kernel, A);
        if (e != cudaSuccess && g_launch_status == cudaSuccess) g_launch_status = e;
        BGSB_LAUNCH_CHECK();
    }
    c->dirty = false;
    c->w = w; c->h = h; c->nimages = nimages; c->last_stream = stream; c->labelled = true;
    c->last_mask = nullptr; c->last_bits = d_bits;
    return BGSB_OK;
}

int ccl_pack_bytes(bgsb_ccl *c, const uint8_t *d_masks, unsigned *d_bits, int w, int h, int nimages, cudaStream_t stream)
{
    BGSB_REQUIRE(c && d_masks && d_bits, "null");
    BGSB_REQUIRE(w > 0 && h > 0 && w <= c->max_w && h <= c->max_h, "image larger than the labeller was created for");
    BGSB_REQUIRE(nimages >= 1 && nimages <= c->max_images, "more images than the labeller was created for");
    BGSB_CUDA(cudaSetDevice(c->device));
    const int wpr = (w + 31) / 32, nwords = wpr * h;
    // (the nodes it creates are replaced by those of the morphology kernel that reads the words)
    launch_pdl(ccl_pack_kernel, dim3((nwords + 255) / 256, nimages), dim3(256), 0, stream, d_masks, d_bits, c->d_parent, w, h,
               wpr, 0, (size_t)w * h, (size_t)nwords);
    BGSB_LAUNCH_CHECK();
    return BGSB_OK;
}

}  // namespace bgsb

using namespace bgsb;

extern "C" {

int bgsb_ccl_create_batch(bgsb_ccl **out, int device, int max_w, int max_h, int max_images)
{
    BGSB_REQUIRE(out, "null out");
    BGSB_REQUIRE(max_w > 0 && max_h > 0 && (long long)max_w * max_h < (1LL << 30), "bad size");
    BGSB_REQUIRE(max_images >= 1 && max_images <= 4096, "max_images out of range");
    BGSB_CUDA(cudaSetDevice(device));
    bgsb_ccl *c = new bgsb_ccl();
    c->device = device; c->max_w = max_w; c->max_h = max_h; c->max_images = max_images;
    c->img_px = (size_t)max_w * max_h;
    c->img_words = (size_t)((max_w + 31) / 32) * max_h;
    c->max_chunks = (int)((c->img_words + 255) / 256);
    // the most 8-connected components an image can hold: isolated pixels on every second row and column
    c->cap = ((max_w + 1) / 2) * ((max_h + 1) / 2) + 64;
    const size_t N = (size_t)max_images;
    cudaError_t e = cudaSuccess;
    auto A = [&](void **p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes); };
    A((void **)&c->d_bits, N * c->img_words * 4);
    A((void **)&c->d_parent, N * c->img_px * 4);
    A((void **)&c->d_outer, N * c->img_px);
    A((void **)&c->d_mask_own, c->img_px);
    A((void **)&c->d_comp, N * (size_t)c->cap * sizeof(CompRaw));
    A((void **)&c->d_ncomp, N * sizeof(int));
    A((void **)&c->d_chunkcount, N * (size_t)c->max_chunks * sizeof(int));
    A((void **)&c->d_chunkprefix, N * (size_t)c->max_chunks * sizeof(int));
    A((void **)&c->d_done, 2 * N * sizeof(int));
    A((void **)&c->d_need_bg, N * sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(c->d_done, 0, 2 * N * sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(c->d_ncomp, 0, N * sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(c->d_comp, 0, N * (size_t)c->cap * sizeof(CompRaw));
    if (e == cudaSuccess) e = cudaMemset(c->d_need_bg, 0, N * sizeof(int));
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        set_error("bgsb_ccl_create: %s", cudaGetErrorString(e));
        bgsb_ccl_destroy(c);
        return BGSB_ERR_CUDA;
    }
    *out = c;
    return BGSB_OK;
}

int bgsb_ccl_create(bgsb_ccl **out, int device, int max_w, int max_h)
{
    return bgsb_ccl_create_batch(out, device, max_w, max_h, 1);
}

void bgsb_ccl_destroy(bgsb_ccl *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    cudaFree(c->d_bits); cudaFree(c->d_parent);
    cudaFree(c->d_outer); cudaFree(c->d_mask_own); cudaFree(c->d_comp); cudaFree(c->d_ncomp);
    cudaFree(c->d_chunkcount); cudaFree(c->d_chunkprefix); cudaFree(c->d_done); cudaFree(c->d_need_bg); cudaFree(c->d_labels_own);
    cudaFree(c->d_rects); cudaFree(c->d_mom);
    if (c->h_pin) cudaFreeHost(c->h_pin);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
}

int bgsb_ccl_label_batch_dev(bgsb_ccl *c, const uint8_t *d_masks, int w, int h, int nimages, int zero_border,
                             int32_t *d_labels, void *stream_)
{
    BGSB_REQUIRE(c && d_masks, "null");
    BGSB_REQUIRE(w > 0 && h > 0 && w <= c->max_w && h <= c->max_h, "image larger than the labeller was created for");
    BGSB_REQUIRE(nimages >= 1 && nimages <= c->max_images, "more images than the labeller was created for");
    BGSB_CUDA(cudaSetDevice(c->device));
    cudaStream_t stream = (cudaStream_t)stream_;
    const int wpr = (w + 31) / 32, nwords = wpr * h;
    const dim3 grid((nwords + 255) / 256, nimages);
    // launch 1: bytes -> bits with the frame already cleared, nodes created (the later launches then run with zero_border = 0)
    launch_pdl(ccl_pack_kernel, grid, dim3(256), 0, stream, d_masks, c->d_bits, c->d_parent, w, h, wpr, zero_border,
               (size_t)w * h, (size_t)nwords);
    BGSB_LAUNCH_CHECK();
    int rc = ccl_label_bits(c, c->d_bits, w, h, nimages, 0, d_labels, stream);
    if (rc) return rc;
    c->last_mask = d_masks; c->last_bits = nullptr;
    return BGSB_OK;
}

int bgsb_ccl_set_param(bgsb_ccl *c, const char *key, double v)
{
    BGSB_REQUIRE(c && key, "null");
    if (std::string(key) == "forceBackgroundPass") c->force_bg = (v != 0);
    else { set_error("bgsb_ccl_set_param: unknown key '%s'", key); return BGSB_ERR_ARG; }
    return BGSB_OK;
}

int bgsb_ccl_label_dev(bgsb_ccl *c, const uint8_t *d_mask, int w, int h, int zero_border, int32_t *d_labels,
                       void *stream_)
{
    return bgsb_ccl_label_batch_dev(c, d_mask, w, h, 1, zero_border, d_labels, stream_);
}

int bgsb_ccl_components_of(bgsb_ccl *c, int image, bgsb_component *out, int capacity, int *n)
{
    BGSB_REQUIRE(c && n, "null");
    if (!c->labelled) { set_error("bgsb_ccl_components: nothing labelled yet"); return BGSB_ERR_STATE; }
    BGSB_REQUIRE(image >= 0 && image < c->nimages, "image index");
    BGSB_CUDA(cudaSetDevice(c->device));
    // one round trip: the count and the first PIN_COMPS rows come back together through pinned memory
    if (!c->h_pin) BGSB_CUDA(cudaMallocHost(&c->h_pin, 64 + (size_t)bgsb_ccl::PIN_COMPS * sizeof(CompRaw)));
    static_assert(sizeof(CompRaw) == sizeof(bgsb_component), "layout");
    const int want = (out && capacity > 0) ? std::min(std::min(capacity, c->cap), (int)bgsb_ccl::PIN_COMPS) : 0;
    BGSB_CUDA(cudaMemcpyAsync(c->h_pin, c->d_ncomp + image, sizeof(int), cudaMemcpyDeviceToHost, c->last_stream));
    if (want)
        BGSB_CUDA(cudaMemcpyAsync(c->h_pin + 64, c->d_comp + (size_t)image * c->cap, (size_t)want * sizeof(CompRaw),
                                  cudaMemcpyDeviceToHost, c->last_stream));
    BGSB_CUDA(cudaStreamSynchronize(c->last_stream));
    const int cnt = *reinterpret_cast<const int *>(c->h_pin);
    *n = cnt;
    if (cnt > c->cap) { set_error("component table overflow (%d > %d)", cnt, c->cap); return BGSB_ERR_CAPACITY; }
    if (!out || capacity <= 0) return BGSB_OK;
    if (cnt > capacity) { set_error("caller table too small (%d > %d)", cnt, capacity); return BGSB_ERR_CAPACITY; }
    if (cnt == 0) return BGSB_OK;
    memcpy(out, c->h_pin + 64, (size_t)std::min(cnt, want) * sizeof(CompRaw));
    if (cnt > want)
        BGSB_CUDA(cudaMemcpy(out + want, c->d_comp + (size_t)image * c->cap + want, (size_t)(cnt - want) * sizeof(CompRaw),
                             cudaMemcpyDeviceToHost));
    for (int i = 0; i < cnt; i++) {       // device rows hold (BIG - xmin, BIG - ymin, xmax, ymax) -> (x, y, w, h)
        out[i].x = CCL_BIG - out[i].x;
        out[i].y = CCL_BIG - out[i].y;
        out[i].w = out[i].w - out[i].x + 1;
        out[i].h = out[i].h - out[i].y + 1;
    }
    return BGSB_OK;
}

int bgsb_ccl_components(bgsb_ccl *c, bgsb_component *out, int capacity, int *n)
{
    return bgsb_ccl_components_of(c, 0, out, capacity, n);
}

int bgsb_ccl_rect_moments_of(bgsb_ccl *c, int image, const int32_t *rects, int nrects, uint64_t *out)
{
    BGSB_REQUIRE(c && out && (rects || nrects == 0), "null");
    if (!c->labelled) { set_error("bgsb_ccl_rect_moments: nothing labelled yet"); return BGSB_ERR_STATE; }
    BGSB_REQUIRE(image >= 0 && image < c->nimages, "image index");
    if (nrects == 0) return BGSB_OK;
    BGSB_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = c->last_stream;
    if (nrects > c->rect_cap) {                              // grows rarely; no allocator calls on the per-frame path
        cudaFree(c->d_rects); cudaFree(c->d_mom); c->d_rects = nullptr; c->d_mom = nullptr; c->rect_cap = 0;
        const int cap = std::max(1024, nrects * 2);
        BGSB_CUDA(cudaMalloc(&c->d_rects, (size_t)cap * 16));
        BGSB_CUDA(cudaMalloc(&c->d_mom, (size_t)cap * 48));
        c->rect_cap = cap;
    }
    if (!c->h_pin) BGSB_CUDA(cudaMallocHost(&c->h_pin, 64 + (size_t)bgsb_ccl::PIN_COMPS * sizeof(CompRaw)));
    const size_t pin_bytes = (size_t)bgsb_ccl::PIN_COMPS * sizeof(CompRaw);
    const bool staged = (size_t)nrects * 48 <= pin_bytes;     // moments come back through pinned memory when they fit
    BGSB_CUDA(cudaMemcpyAsync(c->d_rects, rects, (size_t)nrects * 16, cudaMemcpyHostToDevice, st));
    BGSB_CUDA(cudaMemsetAsync(c->d_mom, 0, (size_t)nrects * 48, st));
    dim3 grid(nrects, 16);
    if (c->last_mask)
        launch_pdl(rect_moments_kernel, dim3(grid), dim3(256), 0, st, c->last_mask + (size_t)image * c->w * c->h, c->w, c->h,
                   c->d_rects, c->d_mom);
    else {
        const int wpr = (c->w + 31) / 32;
        launch_pdl(rect_moments_bits_kernel, dim3(grid), dim3(256), 0, st, c->last_bits + (size_t)image * wpr * c->h, c->w, c->h,
                   wpr, c->d_rects, c->d_mom);
    }
    BGSB_LAUNCH_CHECK();
    BGSB_CUDA(cudaMemcpyAsync(staged ? (void *)(c->h_pin + 64) : (void *)out, c->d_mom, (size_t)nrects * 48,
                              cudaMemcpyDeviceToHost, st));
    BGSB_CUDA(cudaStreamSynchronize(st));
    if (staged) memcpy(out, c->h_pin + 64, (size_t)nrects * 48);
    return BGSB_OK;
}

int bgsb_ccl_rect_moments(bgsb_ccl *c, const int32_t *rects, int nrects, uint64_t *out)
{
    return bgsb_ccl_rect_moments_of(c, 0, rects, nrects, out);
}

int bgsb_ccl_label(bgsb_ccl *c, const uint8_t *mask, int w, int h, size_t stride, int zero_border, int32_t *labels,
                   bgsb_component *out, int capacity, int *n)
{
    BGSB_REQUIRE(c && mask && n, "null");
    BGSB_REQUIRE(stride >= (size_t)w, "stride smaller than a row");
    BGSB_REQUIRE(w > 0 && h > 0 && w <= c->max_w && h <= c->max_h, "image larger than the labeller was created for");
    BGSB_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = c->own_stream;
    BGSB_CUDA(cudaMemcpy2DAsync(c->d_mask_own, w, mask, stride, w, h, cudaMemcpyHostToDevice, st));
    if (labels && !c->d_labels_own) BGSB_CUDA(cudaMalloc(&c->d_labels_own, c->img_px * 4));
    int rc = bgsb_ccl_label_dev(c, c->d_mask_own, w, h, zero_border, labels ? c->d_labels_own : nullptr, st);
    if (rc) return rc;
    if (labels) BGSB_CUDA(cudaMemcpyAsync(labels, c->d_labels_own, (size_t)w * h * 4, cudaMemcpyDeviceToHost, st));
    return bgsb_ccl_components(c, out, capacity, n);
}

}  // extern "C"
