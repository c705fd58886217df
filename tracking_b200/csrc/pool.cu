// Stream pool: N camera streams of one geometry over the GPUs of this process (SURVEY 8e, BASELINE configs 4 / 5).
//
// The reference runs ONE stream per process: its main loop (ustc_src/trackingMain.cpp:161-166) reads a frame and
// pushes it through USTC_BGS::Process, the mask clean-up and the blob detector before it reads the next one;
// FrameProcessor::process (FrameProcessor.cpp:176-195) does the same for the plugin family.  The pool is that loop
// for many cameras: stream s lives on devices[s % ndevices]; every GPU has
//   * one host worker thread that owns the GPU's context work (nothing is enqueued for a GPU from any other thread, so
//     the launch cost of G GPUs is paid in parallel, not G times in a row),
//   * one stream-group pipeline (bgsb_pipeline: plugin -> erode/dilate -> labelling, one launch sequence for all the
//     GPU's streams),
//   * rings of `ring` slots of page-locked host memory for the frames coming in and the masks / component tables
//     going out, and matching device rings, on three CUDA streams (upload / kernels / download) chained by events, so
//     that the upload of slot k+1 overlaps the kernels of slot k and the download of slot k-1.
// Streams never exchange data: no collective, nothing crosses NVLink.
#include <string.h>
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "ccl_internal.h"
#include "kernels.h"

using namespace bgsb;

namespace {

constexpr int POOL_RING_MAX = 8;

// flags: BGSB_POOL_MASKS / BGSB_POOL_DETECT of bgsb_pool_submit; a DETECT job is the moments query of bgsb_pool_detect
struct Job { int slot; int flags; uint64_t seq; bool detect; };

struct GpuGroup {
    int device = 0;
    std::vector<int> streams;                 // global stream ids, in group order
    bgsb_pipeline *pipe = nullptr;
    uint8_t *h_in[POOL_RING_MAX] = {}, *d_in[POOL_RING_MAX] = {};
    uint8_t *h_mask[POOL_RING_MAX] = {}, *d_mask[POOL_RING_MAX] = {};
    int32_t *h_tab[POOL_RING_MAX] = {}, *d_tab[POOL_RING_MAX] = {};
    cudaStream_t s_h2d = nullptr, s_k = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_up[POOL_RING_MAX] = {}, ev_k[POOL_RING_MAX] = {}, ev_done[POOL_RING_MAX] = {};
    bool used[POOL_RING_MAX] = {};
    // worker
    std::thread th;
    std::mutex mu;
    std::condition_variable cv, cv_done;
    std::deque<Job> jobs;
    bool stop = false;
    uint64_t enq_seq[POOL_RING_MAX] = {};      // sequence number of the last job the worker has fully enqueued per slot
    int rc[POOL_RING_MAX] = {};
    int valid[POOL_RING_MAX] = {};
    int has_mask[POOL_RING_MAX] = {};
    int has_dmask[POOL_RING_MAX] = {};        // d_mask[slot] holds the slot's cleaned masks (kept for bgsb_pool_detect)
    std::string err[POOL_RING_MAX];
    // bgsb_pool_detect: the records of this group's streams (filled by the driving thread), their moments query on the
    // worker, on a stream of its own so that it runs beside the next frame sets
    std::vector<MomRec> recs;
    MomentBatch moments;
    cudaStream_t s_det = nullptr;
    cudaEvent_t ev_det = nullptr;
    uint64_t det_seq = 0;                     // sequence number of the last detect job the worker has enqueued
    int det_rc = 0;
    std::string det_err;
};

}  // namespace

struct bgsb_pool {
    int algo = 0, nstreams = 0, w = 0, h = 0, ring = 2, table_rows = 256;
    int zero_border = 1;                             // the pipelines' "zeroBorder"
    int input_format = BGSB_INPUT_BGR;               // "inputFormat": frame_bytes is h*w*3, or h*w*3/2 for YUV 4:2:0
    bool waited[POOL_RING_MAX] = {};                 // the slot's last submit has been waited for
    std::vector<GpuGroup *> groups;
    std::vector<int> group_of, index_in_group;      // per global stream
    uint64_t seq = 0;
    uint64_t want_seq[POOL_RING_MAX] = {};           // sequence number of the last submit per slot
    size_t frame_bytes = 0, mask_bytes = 0, tab_ints = 0;
};

static void worker_main(bgsb_pool *P, GpuGroup *G)
{
    cudaSetDevice(G->device);
    for (;;) {
        Job j;
        {
            std::unique_lock<std::mutex> lk(G->mu);
            G->cv.wait(lk, [&] { return G->stop || !G->jobs.empty(); });
            if (G->jobs.empty()) return;           // stop requested and nothing left to enqueue
            j = G->jobs.front();
            G->jobs.pop_front();
        }
        if (j.detect) {
            // the slot's masks are complete (the caller waited for it) and stay until it is resubmitted
            int rc = G->moments.reserve((int)G->recs.size());
            if (!rc) {
                memcpy(G->moments.h_rec, G->recs.data(), G->recs.size() * sizeof(MomRec));
                rc = G->moments.enqueue(G->d_mask[j.slot], nullptr, P->w, P->h, (int)G->recs.size(), G->s_det);
            }
            if (!rc && cudaEventRecord(G->ev_det, G->s_det) != cudaSuccess) {
                set_error("bgsb_pool_detect: cudaEventRecord -> %s", cudaGetErrorString(cudaGetLastError()));
                rc = BGSB_ERR_CUDA;
            }
            {
                std::lock_guard<std::mutex> lk(G->mu);
                G->det_rc = rc; G->det_err = rc ? bgsb_last_error() : ""; G->det_seq = j.seq;
            }
            G->cv_done.notify_all();
            continue;
        }
        const int k = j.slot;
        const size_t S = G->streams.size();
        int rc = BGSB_OK, valid = 0;
        std::string err;
        auto fail = [&](cudaError_t e, const char *what) {
            if (e != cudaSuccess && rc == BGSB_OK) { rc = BGSB_ERR_CUDA; err = std::string(what) + ": " + cudaGetErrorString(e); (void)cudaGetLastError(); }
            return e != cudaSuccess;
        };
        do {
            // the device input slot was last read by the kernels of its previous use; its outputs by that use's downloads
            if (G->used[k]) {
                if (fail(cudaStreamWaitEvent(G->s_h2d, G->ev_k[k], 0), "wait(kernels of the slot's previous use)")) break;
                if (fail(cudaStreamWaitEvent(G->s_k, G->ev_done[k], 0), "wait(downloads of the slot's previous use)")) break;
            }
            if (fail(cudaMemcpyAsync(G->d_in[k], G->h_in[k], S * P->frame_bytes, cudaMemcpyHostToDevice, G->s_h2d), "upload")) break;
            if (fail(cudaEventRecord(G->ev_up[k], G->s_h2d), "record")) break;
            if (fail(cudaStreamWaitEvent(G->s_k, G->ev_up[k], 0), "wait(upload)")) break;
            int bgv = 0;
            rc = bgsb_pipeline_process_dev(G->pipe, G->d_in[k], P->w, P->h, j.flags ? G->d_mask[k] : nullptr, nullptr, nullptr,
                                           &valid, &bgv, G->s_k);
            if (rc) { err = bgsb_last_error(); break; }
            if (fail(cudaEventRecord(G->ev_k[k], G->s_k), "record")) break;
            if (fail(cudaStreamWaitEvent(G->s_d2h, G->ev_k[k], 0), "wait(kernels)")) break;
            if (valid) {
                // clean-up and labelling run on the pipeline's own stream beside the NEXT frame set's plugin kernel; only
                // the download stream waits for them (masks and tables), the kernel stream goes straight on
                rc = bgsb_pipeline_join_dev(G->pipe, G->s_d2h);
                if (!rc) rc = bgsb_pipeline_tables_dev(G->pipe, G->d_tab[k], P->table_rows, G->s_d2h);
                if (rc) { err = bgsb_last_error(); break; }
            }
            if (valid) {
                if ((j.flags & BGSB_POOL_MASKS) && fail(cudaMemcpyAsync(G->h_mask[k], G->d_mask[k], S * P->mask_bytes, cudaMemcpyDeviceToHost, G->s_d2h), "download masks")) break;
                if (fail(cudaMemcpyAsync(G->h_tab[k], G->d_tab[k], S * P->tab_ints * sizeof(int32_t), cudaMemcpyDeviceToHost, G->s_d2h), "download tables")) break;
            }
            if (fail(cudaEventRecord(G->ev_done[k], G->s_d2h), "record")) break;
            G->used[k] = true;
        } while (0);
        {
            std::lock_guard<std::mutex> lk(G->mu);
            G->rc[k] = rc; G->err[k] = err; G->valid[k] = valid; G->has_mask[k] = valid && (j.flags & BGSB_POOL_MASKS);
            G->has_dmask[k] = valid && j.flags;
            G->enq_seq[k] = j.seq;
        }
        G->cv_done.notify_all();
    }
}

static void pool_free(bgsb_pool *P)
{
    for (GpuGroup *G : P->groups) {
        if (G->th.joinable()) {
            { std::lock_guard<std::mutex> lk(G->mu); G->stop = true; }
            G->cv.notify_all();
            G->th.join();
        }
        cudaSetDevice(G->device);
        cudaDeviceSynchronize();
        if (G->pipe) bgsb_pipeline_destroy(G->pipe);
        for (int k = 0; k < POOL_RING_MAX; k++) {
            if (G->h_in[k]) cudaFreeHost(G->h_in[k]);
            if (G->h_mask[k]) cudaFreeHost(G->h_mask[k]);
            if (G->h_tab[k]) cudaFreeHost(G->h_tab[k]);
            cudaFree(G->d_in[k]); cudaFree(G->d_mask[k]); cudaFree(G->d_tab[k]);
            if (G->ev_up[k]) cudaEventDestroy(G->ev_up[k]);
            if (G->ev_k[k]) cudaEventDestroy(G->ev_k[k]);
            if (G->ev_done[k]) cudaEventDestroy(G->ev_done[k]);
        }
        if (G->s_h2d) cudaStreamDestroy(G->s_h2d);
        if (G->s_k) cudaStreamDestroy(G->s_k);
        if (G->s_d2h) cudaStreamDestroy(G->s_d2h);
        if (G->s_det) cudaStreamDestroy(G->s_det);
        if (G->ev_det) cudaEventDestroy(G->ev_det);
        G->moments.release();
        delete G;
    }
    P->groups.clear();
}

// the table rings at P->table_rows rows per stream (create, and "tableRows" before the first submit)
static int alloc_tables(bgsb_pool *P)
{
    P->tab_ints = (size_t)(P->table_rows + 1) * 8;
    for (GpuGroup *G : P->groups) {
        const size_t bytes = G->streams.size() * P->tab_ints * sizeof(int32_t);
        BGSB_CUDA(cudaSetDevice(G->device));
        for (int k = 0; k < P->ring; k++) {
            if (G->h_tab[k]) cudaFreeHost(G->h_tab[k]);
            cudaFree(G->d_tab[k]);
            G->h_tab[k] = nullptr; G->d_tab[k] = nullptr;
            BGSB_CUDA(cudaHostAlloc((void **)&G->h_tab[k], bytes, cudaHostAllocDefault));
            BGSB_CUDA(cudaMalloc(&G->d_tab[k], bytes));
        }
    }
    return BGSB_OK;
}

// the frame rings at P->frame_bytes per stream ("inputFormat" before the first submit)
static int alloc_frames(bgsb_pool *P)
{
    for (GpuGroup *G : P->groups) {
        const size_t bytes = G->streams.size() * P->frame_bytes;
        BGSB_CUDA(cudaSetDevice(G->device));
        for (int k = 0; k < P->ring; k++) {
            if (G->h_in[k]) cudaFreeHost(G->h_in[k]);
            cudaFree(G->d_in[k]);
            G->h_in[k] = nullptr; G->d_in[k] = nullptr;
            BGSB_CUDA(cudaHostAlloc((void **)&G->h_in[k], bytes, cudaHostAllocDefault));
            BGSB_CUDA(cudaMalloc(&G->d_in[k], bytes));
        }
    }
    return BGSB_OK;
}

extern "C" {

int bgsb_pool_create(bgsb_pool **out, int algo, int nstreams, const int *devices, int ndevices, int w, int h, int ring)
{
    BGSB_REQUIRE(out && devices, "null");
    BGSB_REQUIRE(nstreams >= 1 && ndevices >= 1 && ndevices <= 64, "nstreams >= 1, 1 <= ndevices <= 64");
    BGSB_REQUIRE(w > 0 && h > 0 && (long long)w * h < (1LL << 27), "bad geometry");
    BGSB_REQUIRE(ring >= 1 && ring <= POOL_RING_MAX, "ring in [1,8]");
    bgsb_pool *P = new bgsb_pool();
    P->algo = algo; P->nstreams = nstreams; P->w = w; P->h = h; P->ring = ring;
    P->frame_bytes = (size_t)w * h * 3; P->mask_bytes = (size_t)w * h;
    P->group_of.assign(nstreams, 0); P->index_in_group.assign(nstreams, 0);
    const int ng = std::min(ndevices, nstreams);
    int rc = BGSB_OK;
    for (int g = 0; g < ng && rc == BGSB_OK; g++) {
        GpuGroup *G = new GpuGroup();
        P->groups.push_back(G);
        G->device = devices[g];
        for (int s = g; s < nstreams; s += ng) {           // stream s -> GPU s mod G
            P->group_of[s] = g; P->index_in_group[s] = (int)G->streams.size();
            G->streams.push_back(s);
        }
        const size_t S = G->streams.size();
        cudaError_t e = cudaSetDevice(G->device);
        if (e == cudaSuccess) rc = bgsb_pipeline_create(&G->pipe, algo, G->device, (int)S);
        if (rc) break;
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&G->s_h2d, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&G->s_k, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&G->s_d2h, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&G->s_det, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&G->ev_det, cudaEventDisableTiming);
        for (int k = 0; k < ring && e == cudaSuccess; k++) {
            e = cudaHostAlloc((void **)&G->h_in[k], S * P->frame_bytes, cudaHostAllocDefault);
            if (e == cudaSuccess) e = cudaHostAlloc((void **)&G->h_mask[k], S * P->mask_bytes, cudaHostAllocDefault);
            if (e == cudaSuccess) e = cudaMalloc(&G->d_in[k], S * P->frame_bytes);
            if (e == cudaSuccess) e = cudaMalloc(&G->d_mask[k], S * P->mask_bytes);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&G->ev_up[k], cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&G->ev_k[k], cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&G->ev_done[k], cudaEventDisableTiming);
        }
        if (e != cudaSuccess) {
            set_error("bgsb_pool_create (device %d, %zu streams): %s", G->device, S, cudaGetErrorString(e));
            (void)cudaGetLastError();
            rc = BGSB_ERR_CUDA;
        }
    }
    if (!rc) rc = alloc_tables(P);
    if (rc) { pool_free(P); delete P; return rc; }
    for (GpuGroup *G : P->groups) G->th = std::thread(worker_main, P, G);
    *out = P;
    return BGSB_OK;
}

void bgsb_pool_destroy(bgsb_pool *P)
{
    if (!P) return;
    pool_free(P);
    delete P;
}

int bgsb_pool_set_param(bgsb_pool *P, const char *key, double v)
{
    BGSB_REQUIRE(P && key, "null");
    if (std::string(key) == "tableRows") {
        BGSB_REQUIRE(P->seq == 0, "tableRows: set it before the first submit");
        BGSB_REQUIRE(v >= 1 && v <= (1 << 24), "tableRows in [1, 2^24]");
        P->table_rows = (int)v;
        return alloc_tables(P);
    }
    if (std::string(key) == "inputFormat") {
        BGSB_REQUIRE(P->seq == 0, "inputFormat: set it before the first submit");
        BGSB_REQUIRE(v == BGSB_INPUT_BGR || v == BGSB_INPUT_NV12 || v == BGSB_INPUT_I420,
                     "inputFormat is 0 (BGSB_INPUT_BGR), 1 (BGSB_INPUT_NV12) or 2 (BGSB_INPUT_I420)");
        BGSB_REQUIRE(v == BGSB_INPUT_BGR || (P->w % 2 == 0 && P->h % 2 == 0),
                     "YUV 4:2:0 input (inputFormat NV12 / I420) needs an even width and height");
        for (GpuGroup *G : P->groups) {
            int rc = bgsb_pipeline_set_param(G->pipe, key, v);
            if (rc) return rc;
        }
        P->input_format = (int)v;
        const size_t npx = (size_t)P->w * P->h, fb = v == BGSB_INPUT_BGR ? npx * 3 : npx * 3 / 2;
        if (fb == P->frame_bytes) return BGSB_OK;
        P->frame_bytes = fb;
        return alloc_frames(P);
    }
    for (GpuGroup *G : P->groups) {
        int rc = bgsb_pipeline_set_param(G->pipe, key, v);
        if (rc) return rc;
    }
    if (std::string(key) == "zeroBorder") P->zero_border = (v != 0);
    return BGSB_OK;
}

int bgsb_pool_set_morph(bgsb_pool *P, const int *ops, int nops)
{
    BGSB_REQUIRE(P, "null");
    for (GpuGroup *G : P->groups) {
        int rc = bgsb_pipeline_set_morph(G->pipe, ops, nops);
        if (rc) return rc;
    }
    return BGSB_OK;
}

int bgsb_pool_device_of(bgsb_pool *P, int stream, int *device)
{
    BGSB_REQUIRE(P && device && stream >= 0 && stream < P->nstreams, "stream index");
    *device = P->groups[P->group_of[stream]]->device;
    return BGSB_OK;
}

uint8_t *bgsb_pool_frame_buffer(bgsb_pool *P, int stream, int slot)
{
    if (!P || stream < 0 || stream >= P->nstreams || slot < 0 || slot >= P->ring) return nullptr;
    GpuGroup *G = P->groups[P->group_of[stream]];
    return G->h_in[slot] + (size_t)P->index_in_group[stream] * P->frame_bytes;
}

int bgsb_pool_submit(bgsb_pool *P, int slot, int flags)
{
    BGSB_REQUIRE(P && slot >= 0 && slot < P->ring, "slot index");
    BGSB_REQUIRE((flags & ~(BGSB_POOL_MASKS | BGSB_POOL_DETECT)) == 0, "flags: BGSB_POOL_MASKS | BGSB_POOL_DETECT");
    const uint64_t seq = ++P->seq;
    P->want_seq[slot] = seq;
    P->waited[slot] = false;
    for (GpuGroup *G : P->groups) {
        { std::lock_guard<std::mutex> lk(G->mu); G->jobs.push_back(Job{slot, flags, seq, false}); }
        G->cv.notify_one();
    }
    return BGSB_OK;
}

int bgsb_pool_wait(bgsb_pool *P, int slot, int *valid)
{
    BGSB_REQUIRE(P && slot >= 0 && slot < P->ring, "slot index");
    if (valid) *valid = 0;
    if (P->want_seq[slot] == 0) { set_error("bgsb_pool_wait: nothing was submitted for slot %d", slot); return BGSB_ERR_STATE; }
    int all_valid = 1;
    for (GpuGroup *G : P->groups) {
        {
            std::unique_lock<std::mutex> lk(G->mu);
            G->cv_done.wait(lk, [&] { return G->enq_seq[slot] >= P->want_seq[slot]; });
            if (G->rc[slot]) { set_error("bgsb_pool (device %d): %s", G->device, G->err[slot].c_str()); return G->rc[slot]; }
            all_valid &= G->valid[slot];
        }
        BGSB_CUDA(cudaEventSynchronize(G->ev_done[slot]));
    }
    P->waited[slot] = true;
    if (valid) *valid = all_valid;
    return BGSB_OK;
}

const uint8_t *bgsb_pool_mask(bgsb_pool *P, int stream, int slot)
{
    if (!P || stream < 0 || stream >= P->nstreams || slot < 0 || slot >= P->ring) return nullptr;
    GpuGroup *G = P->groups[P->group_of[stream]];
    if (!G->has_mask[slot]) return nullptr;
    return G->h_mask[slot] + (size_t)P->index_in_group[stream] * P->mask_bytes;
}

int bgsb_pool_components(bgsb_pool *P, int stream, int slot, bgsb_component *out, int capacity, int *n)
{
    BGSB_REQUIRE(P && n && stream >= 0 && stream < P->nstreams && slot >= 0 && slot < P->ring, "bad args");
    GpuGroup *G = P->groups[P->group_of[stream]];
    if (!G->valid[slot]) { *n = 0; set_error("bgsb_pool_components: the slot holds no mask (plugin warm-up frame)"); return BGSB_ERR_STATE; }
    const int32_t *t = G->h_tab[slot] + (size_t)P->index_in_group[stream] * P->tab_ints;
    const int cnt = t[0];
    *n = cnt;
    if (!out || capacity <= 0) return BGSB_OK;
    if (cnt > capacity) { set_error("caller table too small (%d > %d)", cnt, capacity); return BGSB_ERR_CAPACITY; }
    if (cnt > P->table_rows) {
        set_error("stream %d has %d components, the pool keeps the first %d per frame (noisy mask?)", stream, cnt, P->table_rows);
        memcpy(out, t + 8, (size_t)P->table_rows * sizeof(bgsb_component));
        return BGSB_ERR_CAPACITY;
    }
    memcpy(out, t + 8, (size_t)cnt * sizeof(bgsb_component));
    return BGSB_OK;
}

int bgsb_pool_detect(bgsb_pool *P, int slot, bgsb_blobdetector *const *bds, const bgsb_blob *const *old_blobs,
                     const int *n_old, bgsb_blob *new_blobs, int *result, bgsb_blob *frame_blobs, int *n_frame, int *status)
{
    BGSB_REQUIRE(P && slot >= 0 && slot < P->ring, "slot index");
    BGSB_REQUIRE(new_blobs && result && status, "null");
    if (!P->waited[slot]) { set_error("bgsb_pool_detect: slot %d has not been waited for since its submit", slot); return BGSB_ERR_STATE; }
    for (GpuGroup *G : P->groups) {
        if (!G->valid[slot]) { set_error("bgsb_pool_detect: the slot holds no mask (plugin warm-up frame)"); return BGSB_ERR_STATE; }
        if (!G->has_dmask[slot]) {
            set_error("bgsb_pool_detect: slot %d was submitted without BGSB_POOL_DETECT", slot);
            return BGSB_ERR_STATE;
        }
    }
    int rc = detect_check(bds, P->nstreams, old_blobs, n_old, P->zero_border);
    if (rc) return rc;
    // (a) per stream from the tables on the host; the rectangles of a GPU's streams go to its worker as one query
    const int N = P->nstreams;
    std::vector<std::vector<int32_t>> rects(N);
    int over = -1;
    for (int s = 0; s < N; s++) {
        GpuGroup *G = P->groups[P->group_of[s]];
        const int32_t *t = G->h_tab[slot] + (size_t)P->index_in_group[s] * P->tab_ints;
        status[s] = t[0] > P->table_rows ? BGSB_ERR_CAPACITY : BGSB_OK;
        if (status[s]) { if (over < 0) over = s; continue; }
        detect_rects(bds[s], reinterpret_cast<const bgsb_component *>(t + 8), t[0], P->w, P->h, rects[s]);
    }
    std::vector<int> first(N, 0);
    for (GpuGroup *G : P->groups) {
        G->recs.clear();
        for (int s : G->streams) {
            first[s] = (int)G->recs.size();
            const std::vector<int32_t> &r = rects[s];
            for (size_t i = 0; i < r.size(); i += 4)
                G->recs.push_back(MomRec{P->index_in_group[s], r[i], r[i + 1], r[i + 2], r[i + 3], 0, 0, 0});
        }
    }
    const uint64_t seq = ++P->seq;
    for (GpuGroup *G : P->groups) {
        { std::lock_guard<std::mutex> lk(G->mu); G->jobs.push_back(Job{slot, 0, seq, true}); }
        G->cv.notify_one();
    }
    for (GpuGroup *G : P->groups) {
        std::unique_lock<std::mutex> lk(G->mu);
        G->cv_done.wait(lk, [&] { return G->det_seq >= seq; });
        if (G->det_rc && !rc) { rc = G->det_rc; set_error("bgsb_pool_detect (device %d): %s", G->device, G->det_err.c_str()); }
    }
    if (rc) return rc;
    for (GpuGroup *G : P->groups) BGSB_CUDA(cudaEventSynchronize(G->ev_det));
    // (b) per stream
    for (int s = 0; s < N; s++) {
        if (status[s]) continue;
        GpuGroup *G = P->groups[P->group_of[s]];
        int n_new = 0;
        detect_finish(bds[s], rects[s].data(), (int)rects[s].size() / 4,
                      reinterpret_cast<const uint64_t *>(G->moments.h_mom) + 6 * first[s], P->w, P->h,
                      old_blobs ? old_blobs[s] : nullptr, old_blobs ? n_old[s] : 0, new_blobs + s, 1, &n_new, result + s,
                      frame_blobs ? frame_blobs + 10 * s : nullptr, 10, n_frame ? n_frame + s : nullptr);
    }
    if (over >= 0) {
        set_error("bgsb_pool_detect: stream %d (and maybe others) has more components than \"tableRows\" = %d; its "
                  "detector did not advance", over, P->table_rows);
        return BGSB_ERR_CAPACITY;
    }
    return BGSB_OK;
}

int bgsb_pool_info(bgsb_pool *P, int *ngroups, int *ring, int *table_rows)
{
    BGSB_REQUIRE(P, "null");
    if (ngroups) *ngroups = (int)P->groups.size();
    if (ring) *ring = P->ring;
    if (table_rows) *table_rows = P->table_rows;
    return BGSB_OK;
}

}  // extern "C"
