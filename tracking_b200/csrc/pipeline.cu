// The foreground pipeline as one device-resident object per group of camera streams:
//
//     IBGS::process  ->  mask clean-up (erode / dilate chain)  ->  steps 1-2 of CvBlobDetectorCC::DetectNewBlob
//
// which is what the reference's main loop does once per frame and stream (ustc_src/trackingMain.cpp:161-166:
// cvQueryFrame, then CvBlobTrackerAuto1::Process = USTC_BGS::Process (ustc_src/ustc_bgs.cpp:87-113, the plugin),
// the FG post-processing and CvBlobDetectorCC::DetectNewBlob (:626), SURVEY 3.1 / 8a rows a1-aC).
//
// Between the stages the mask stays BIT-PACKED (32 pixels per word): the MOG2 kernel sets the bits of its foreground
// pixels directly (its fast path never produces foreground, so only the generic phase touches the words), the
// morphology kernel reads and writes words and also creates the labeller's union-find nodes, and the labeller starts at
// its merge step.  Per frame of the whole stream group: one memset of the packed rows, the plugin kernel, the
// morphology kernel and three labelling launches -- against 1 + 1 + 12 launches and three byte<->bit conversions
// when the same stages are chained through the byte-mask entry points.  Byte masks ({0,255}) are produced only when
// the caller asks for them (they are the host-boundary format of IBGS / CvFGDetector::GetMask).
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <string>

#include <nvtx3/nvToolsExt.h>

#include "ccl_internal.h"
#include "kernels.h"

using namespace bgsb;

struct bgsb_pipeline {
    int device = 0, nstreams = 1;
    bgsb_ctx *bgs = nullptr;
    bgsb_ccl *ccl = nullptr;
    int ops[32];
    int nops = 0, total_iters = 0;
    int zero_border = 1;              // OpenCV 2.4 cvFindContours (the version the reference builds against)
    int force_bg = 0;
    int chain_ctas = 0;               // > 0: background pass as plain launches of at most this many CTAs (0: cooperative)
    int w = 0, h = 0;
    static constexpr int NSLOT = 4;                     // plugin-mask buffers in rotation: the chain of frame t may still be
                                                        // reading its buffer while the plugin kernels of t+1 .. t+3 run
    unsigned *d_raw[NSLOT] = {};                        // [S][h][wpr] packed plugin masks
    unsigned *d_clean = nullptr;                        // ... after the chain
    uint8_t *d_fg[NSLOT] = {};                          // [S][h][w] byte masks of plugins that cannot emit bits
    bool labelled = false;
    bool raw_chain = false;                             // the last labelled frame: threshold off, chain on (no moments)
    // Clean-up + labelling of frame t run on the pipeline's own high-priority stream, so that they overlap the plugin
    // kernel of frame t+1 (their launches are latency-bound and leave the SMs almost empty): the caller's stream only
    // waits for them when it has to (device outputs requested, or bgsb_pipeline_join_dev).
    cudaStream_t side = nullptr;
    cudaEvent_t ev_plugin = nullptr, ev_chain[NSLOT] = {}, ev_out = nullptr;
    bool chain_used[NSLOT] = {};
    uint64_t nframe = 0;
    int last_slot = -1;                                 // slot of the last frame whose chain was enqueued, -1: none
};

static void pipeline_free(bgsb_pipeline *p)
{
    for (int i = 0; i < bgsb_pipeline::NSLOT; i++) { cudaFree(p->d_raw[i]); cudaFree(p->d_fg[i]); p->d_raw[i] = nullptr; p->d_fg[i] = nullptr; p->chain_used[i] = false; }
    cudaFree(p->d_clean); p->d_clean = nullptr;
    p->last_slot = -1;
    if (p->ccl) { bgsb_ccl_destroy(p->ccl); p->ccl = nullptr; }
    p->w = p->h = 0; p->labelled = false;
}

static int pipeline_geometry(bgsb_pipeline *p, int w, int h)
{
    if (p->w == w && p->h == h) return BGSB_OK;
    pipeline_free(p);
    const size_t S = (size_t)p->nstreams, words = (size_t)((w + 31) / 32) * h;
    if (p->side) cudaStreamSynchronize(p->side);
    cudaError_t e = cudaMalloc(&p->d_clean, S * words * 4);
    for (int i = 0; i < bgsb_pipeline::NSLOT && e == cudaSuccess; i++) {
        e = cudaMalloc(&p->d_raw[i], S * words * 4);
        if (e == cudaSuccess) e = cudaMemset(p->d_raw[i], 0, S * words * 4);
    }
    if (e == cudaSuccess && !p->side) {
        int lo = 0, hi = 0;
        e = cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&p->side, cudaStreamNonBlocking, hi);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_plugin, cudaEventDisableTiming);
        for (int i = 0; i < bgsb_pipeline::NSLOT && e == cudaSuccess; i++) e = cudaEventCreateWithFlags(&p->ev_chain[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_out, cudaEventDisableTiming);
    }
    if (e != cudaSuccess) {
        set_error("bgsb_pipeline(%d x %d x %d streams): %s", w, h, p->nstreams, cudaGetErrorString(e));
        (void)cudaGetLastError();
        pipeline_free(p);
        return BGSB_ERR_CUDA;
    }
    int rc = bgsb_ccl_create_batch(&p->ccl, p->device, w, h, p->nstreams);
    if (rc) { pipeline_free(p); return rc; }
    p->w = w; p->h = h;
    return BGSB_OK;
}

extern "C" {

int bgsb_pipeline_create(bgsb_pipeline **out, int algo, int device, int nstreams)
{
    BGSB_REQUIRE(out, "null out");
    bgsb_ctx *bgs = nullptr;
    int rc = bgsb_create_group(&bgs, algo, device, nstreams);
    if (rc) return rc;
    bgsb_pipeline *p = new bgsb_pipeline();
    p->device = device; p->nstreams = nstreams; p->bgs = bgs;
    p->ops[0] = BGSB_MORPH_ERODE; p->ops[1] = 1; p->ops[2] = BGSB_MORPH_DILATE; p->ops[3] = 1;     // OPEN 3x3 (SURVEY 8a row aM)
    p->nops = 2; p->total_iters = 2;
    *out = p;
    return BGSB_OK;
}

void bgsb_pipeline_destroy(bgsb_pipeline *p)
{
    if (!p) return;
    cudaSetDevice(p->device);
    cudaDeviceSynchronize();
    pipeline_free(p);
    if (p->side) cudaStreamDestroy(p->side);
    if (p->ev_plugin) cudaEventDestroy(p->ev_plugin);
    for (int i = 0; i < bgsb_pipeline::NSLOT; i++) if (p->ev_chain[i]) cudaEventDestroy(p->ev_chain[i]);
    if (p->ev_out) cudaEventDestroy(p->ev_out);
    bgsb_destroy(p->bgs);
    delete p;
}

bgsb_ctx *bgsb_pipeline_bgs(bgsb_pipeline *p) { return p ? p->bgs : nullptr; }

int bgsb_pipeline_set_morph(bgsb_pipeline *p, const int *ops, int nops)
{
    BGSB_REQUIRE(p && nops >= 0 && nops <= 16 && (nops == 0 || ops), "at most 16 (op, iterations) pairs");
    int total = 0;
    for (int i = 0; i < nops; i++) {
        BGSB_REQUIRE(ops[2 * i] == BGSB_MORPH_ERODE || ops[2 * i] == BGSB_MORPH_DILATE, "bad op");
        BGSB_REQUIRE(ops[2 * i + 1] >= 0 && ops[2 * i + 1] <= 64, "iterations out of range");
        total += ops[2 * i + 1];
    }
    memcpy(p->ops, ops, sizeof(int) * 2 * nops);
    p->nops = nops; p->total_iters = total;
    return BGSB_OK;
}

int bgsb_pipeline_set_param(bgsb_pipeline *p, const char *key, double v)
{
    BGSB_REQUIRE(p && key, "null");
    const std::string k(key);
    if (k == "zeroBorder") p->zero_border = (v != 0);
    else if (k == "chainCtas") { BGSB_REQUIRE(v >= 0 && v <= 1e6, "chainCtas >= 0"); p->chain_ctas = (int)v; }
    else if (k == "forceBackgroundPass") { p->force_bg = (v != 0); if (p->ccl) p->ccl->force_bg = p->force_bg; }
    else return bgsb_set_param(p->bgs, key, v);
    return BGSB_OK;
}

int bgsb_pipeline_process_dev(bgsb_pipeline *p, const uint8_t *d_frames, int w, int h, uint8_t *d_mask, uint8_t *d_bg,
                              int32_t *d_labels, int *valid, int *bg_valid, void *stream_)
{
    BGSB_REQUIRE(p && d_frames, "null");
    BGSB_REQUIRE(w > 0 && h > 0, "empty frame");
    BGSB_CUDA(cudaSetDevice(p->device));
    cudaStream_t stream = (cudaStream_t)stream_;
    if (valid) *valid = 0;
    nvtxRangePushA("bgsb_pipeline: plugin + clean-up + labelling");
    struct NvtxPop { ~NvtxPop() { nvtxRangePop(); } } nvtx_pop;
    int rc = pipeline_geometry(p, w, h);
    if (rc) return rc;
    p->ccl->force_bg = p->force_bg;
    // "chainCtas" > 0: the labeller's background pass as four plain launches of at most that many CTAs instead of one
    // cooperative launch (which has to become resident as a whole beside the next frame set's plugin kernel); measured,
    // the cooperative form is the faster one (8 x 1080p streams 218 vs 225 us per frame set) and stays the default
    p->ccl->max_ctas = p->chain_ctas;
    const int S = p->nstreams;
    const size_t words = (size_t)((w + 31) / 32) * h;
    // Packed output needs a {0,255} mask: with the plugin's threshold off and no chain, DetectNewBlob's moments weigh the
    // raw mask values (shadow = 127), so that combination keeps the byte mask.
    double thr_on = 1.;
    (void)bgsb_get_param(p->bgs, "enableThreshold", &thr_on);
    // With the threshold off and a chain, the reference erodes / dilates the raw grey-level mask and DetectNewBlob then
    // keeps the pixels > 128.  Thresholding commutes with erode / dilate (min / max), so packing "> 128" BEFORE the chain
    // labels the same pixels; the cleaned grey-level mask and its moments would need grey-level morphology, so they are
    // refused in that combination.
    const bool raw_chain = thr_on == 0. && p->total_iters > 0;
    if (raw_chain && d_mask) {
        set_error("bgsb_pipeline_process_dev: no cleaned mask with enableThreshold = 0 and an erode / dilate chain (the "
                  "reference's is grey-level); pass d_mask = NULL");
        return BGSB_ERR_ARG;
    }
    const bool pack = ctx_can_pack(p->bgs) && (p->total_iters > 0 || thr_on != 0.);
    const int slot = (int)(p->nframe % bgsb_pipeline::NSLOT);
    if (!pack && !p->d_fg[slot]) BGSB_CUDA(cudaMalloc(&p->d_fg[slot], (size_t)S * w * h));
    // this slot's plugin mask was last read by the chain of the frame NSLOT frames ago
    if (p->chain_used[slot]) BGSB_CUDA(cudaStreamWaitEvent(stream, p->ev_chain[slot], 0));
    int packed = 0, fv = 0, bv = 0;
    if (pack) {
        // the plugin kernel ORs its foreground bits into zeroed rows; a pixel counts when its mask byte is > 128 (what
        // cvThreshold(128) in DetectNewBlob keeps; on a thresholded {0,255} mask the same as non-zero, which is what the
        // morphology reads)
        // (the rows are zero: cleared at allocation and, after every use, behind the chain that read them)
        rc = ctx_process_frame(p->bgs, d_frames, w, h, nullptr, d_bg, p->d_raw[slot], 128, &packed, &fv, &bv, stream);
    } else {
        rc = ctx_process_frame(p->bgs, d_frames, w, h, p->d_fg[slot], d_bg, nullptr, 0, &packed, &fv, &bv, stream);
    }
    if (rc) return rc;
    if (bg_valid) *bg_valid = bv;
    if (!fv) return BGSB_OK;                       // FD frame 0 / WMV frames 0-1: no mask yet (reference early returns)
    p->nframe++;
    // ---- clean-up + labelling on the side stream ----
    cudaStream_t cs = p->side;
    BGSB_CUDA(cudaEventRecord(p->ev_plugin, stream));
    BGSB_CUDA(cudaStreamWaitEvent(cs, p->ev_plugin, 0));
    MorphIO io;
    memset(&io, 0, sizeof(io));
    io.parent = p->ccl->d_parent; io.zero_border = p->zero_border;
    io.out_bytes = d_mask;
    if (packed) {
        // (an empty chain still goes through the kernel: it copies the rows to d_clean -- the plugin's rows are cleared
        // below for their next use -- and creates the labeller's nodes)
        io.in_bits = p->d_raw[slot]; io.out_bits = p->d_clean;
        rc = launch_morph_chain_io(io, w, h, S, p->ops, p->nops, cs);
        if (rc) return rc;
        rc = ccl_label_bits(p->ccl, p->d_clean, w, h, S, p->zero_border, d_labels, cs);
    } else if (raw_chain) {
        // raw grey-level mask: DetectNewBlob's threshold first (the labeller's pack step), then the chain on the words
        rc = ccl_pack_bytes(p->ccl, p->d_fg[slot], p->d_raw[slot], w, h, S, cs);
        if (rc) return rc;
        io.in_bits = p->d_raw[slot]; io.out_bits = p->d_clean;
        rc = launch_morph_chain_io(io, w, h, S, p->ops, p->nops, cs);
        if (rc) return rc;
        rc = ccl_label_bits(p->ccl, p->d_clean, w, h, S, p->zero_border, d_labels, cs);
    } else if (p->total_iters > 0) {
        io.in_bytes = p->d_fg[slot]; io.out_bits = p->d_clean;
        rc = launch_morph_chain_io(io, w, h, S, p->ops, p->nops, cs);
        if (rc) return rc;
        rc = ccl_label_bits(p->ccl, p->d_clean, w, h, S, p->zero_border, d_labels, cs);
    } else {
        // no chain on a byte mask: the labeller's own pack step applies DetectNewBlob's threshold (> 128)
        if (d_mask) BGSB_CUDA(cudaMemcpyAsync(d_mask, p->d_fg[slot], (size_t)S * w * h, cudaMemcpyDeviceToDevice, cs));
        rc = bgsb_ccl_label_batch_dev(p->ccl, p->d_fg[slot], w, h, S, p->zero_border, d_labels, cs);
    }
    if (rc) return rc;
    if (packed) BGSB_CUDA(cudaMemsetAsync(p->d_raw[slot], 0, S * words * 4, cs));    // ready for the plugin two frames on
    BGSB_CUDA(cudaEventRecord(p->ev_chain[slot], cs));
    p->chain_used[slot] = true;
    p->last_slot = slot;
    // device outputs the caller may consume on its stream: that stream waits for them now; table-only frames leave the
    // chain running beside whatever the caller enqueues next (the next frame's plugin kernel)
    if (d_mask || d_labels) BGSB_CUDA(cudaStreamWaitEvent(stream, p->ev_chain[slot], 0));
    p->labelled = true;
    p->raw_chain = raw_chain;
    if (valid) *valid = 1;
    return BGSB_OK;
}

int bgsb_pipeline_join_dev(bgsb_pipeline *p, void *stream)
{
    BGSB_REQUIRE(p, "null");
    BGSB_CUDA(cudaSetDevice(p->device));
    if (p->last_slot >= 0) BGSB_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, p->ev_chain[p->last_slot], 0));
    return BGSB_OK;
}

int bgsb_pipeline_components(bgsb_pipeline *p, int stream_index, bgsb_component *out, int capacity, int *n)
{
    BGSB_REQUIRE(p && n, "null");
    if (!p->labelled) { set_error("bgsb_pipeline_components: no frame has produced a mask yet"); return BGSB_ERR_STATE; }
    return bgsb_ccl_components_of(p->ccl, stream_index, out, capacity, n);
}

int bgsb_pipeline_tables_dev(bgsb_pipeline *p, int32_t *d_out, int rows_per_stream, void *stream)
{
    BGSB_REQUIRE(p && d_out && rows_per_stream >= 0, "bad args");
    if (!p->labelled) { set_error("bgsb_pipeline_tables_dev: no frame has produced a mask yet"); return BGSB_ERR_STATE; }
    BGSB_CUDA(cudaSetDevice(p->device));
    int rc = ccl_gather_tables(p->ccl, d_out, rows_per_stream, p->side);       // behind the labelling, on its stream
    if (rc) return rc;
    BGSB_CUDA(cudaEventRecord(p->ev_out, p->side));
    BGSB_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, p->ev_out, 0));
    return BGSB_OK;
}

int bgsb_pipeline_rect_moments(bgsb_pipeline *p, int stream_index, const int32_t *rects, int nrects, uint64_t *out)
{
    BGSB_REQUIRE(p && out, "null");
    if (!p->labelled) { set_error("bgsb_pipeline_rect_moments: no frame has produced a mask yet"); return BGSB_ERR_STATE; }
    if (p->raw_chain) {
        set_error("bgsb_pipeline_rect_moments: with enableThreshold = 0 and an erode / dilate chain the reference weighs the "
                  "grey-level cleaned mask, which the pipeline does not compute");
        return BGSB_ERR_ARG;
    }
    return bgsb_ccl_rect_moments_of(p->ccl, stream_index, rects, nrects, out);
}

}  // extern "C"
