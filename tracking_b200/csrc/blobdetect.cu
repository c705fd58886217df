// CvBlobDetectorCC replacement: connected components + sums on the GPU (ccl.cu), list logic on the host.
//
// Replaces CvBlobDetectorCC::DetectNewBlob of OpenCV 2.4 `legacy` (cvCreateBlobDetectorCC), which the
// reference plugs into its pipeline at ustc_src/trackingMain.cpp:56 (module table) and :626 (creation),
// listed as stage "BlobDetector" in readme.md:4-10.  OpenCV legacy is an external dependency that is not
// vendored in the reference tree; this file follows the restated specification of SURVEY.md Appendix A.6:
//   1-2  threshold 128 + external contours         -> bgsb_ccl (GPU)
//   3    cvSeqPartition of contour rects (CompareContour)      -> partition_rects()
//   4    union rect per cluster, cvMoments of the mask inside it -> bgsb_ccl_rect_moments (GPU sums)
// Steps 3 and 5-7 are detect_rects (before the moments) and detect_finish (after them); bgsb_pipeline_detect and
// bgsb_pool_detect run them around one moments launch for all their streams.
//   5    drop small blobs and blobs overlapping tracked ones
//   6    insertion sort by w*h (descending), keep 10
//   7    track lists over the last `Latency` frames, uniform-motion test, emit best new blob
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <vector>

#include "ccl_internal.h"

using namespace bgsb;

namespace {

constexpr int SEQ_SIZE_MAX = 30;
constexpr int SEQ_NUM = 1000;

struct Track {
    int size = 0;
    bool has[SEQ_SIZE_MAX];
    bgsb_blob blobs[SEQ_SIZE_MAX];
    Track() { memset(has, 0, sizeof(has)); memset(blobs, 0, sizeof(blobs)); }
};

struct Rect { int x, y, w, h; };

// CompareContour (legacy/enteringblobdetection.cpp): rects are "equal" when they overlap in x
// and their vertical gap is below 0.3 * the taller height.  fp32 as in the original.
inline bool rects_close(const Rect &ra, const Rect &rb)
{
    float pax = ra.x + ra.w * 0.5f, pay = ra.y + ra.h * 0.5f;
    float pbx = rb.x + rb.w * 0.5f, pby = rb.y + rb.h * 0.5f;
    float w = (ra.w + rb.w) * 0.5f, h = (ra.h + rb.h) * 0.5f;
    float dx = (float)(fabs(pax - pbx) - w);
    float dy = (float)(fabs(pay - pby) - h);
    float wt = 0;
    float ht = std::max(ra.h, rb.h) * 0.3f;
    return dx < wt && dy < ht;
}

// cvSeqPartition: transitive closure of the predicate; classes numbered by first appearance.
// cvSeqPartition itself tests all n(n-1)/2 pairs.  The predicate needs the x-extents to overlap (dx < 0), so
// only pairs whose integer x-ranges come within one pixel of each other can satisfy it: a sweep over the
// rectangles sorted by x hands exactly those pairs to the exact float predicate.  The partition and its
// numbering (first member of each class in index order) do not depend on the order the pairs are visited in.
int partition_rects(const std::vector<Rect> &r, std::vector<int> &cls)
{
    const int n = (int)r.size();
    std::vector<int> parent(n);
    for (int i = 0; i < n; i++) parent[i] = i;
    auto find = [&](int a) { while (parent[a] != a) { parent[a] = parent[parent[a]]; a = parent[a]; } return a; };
    std::vector<int> order(n);
    for (int i = 0; i < n; i++) order[i] = i;
    std::sort(order.begin(), order.end(), [&](int a, int b) { return r[a].x < r[b].x; });
    for (int u = 0; u < n; u++) {
        const int i = order[u];
        const int xend = r[i].x + r[i].w + 1;
        for (int v = u + 1; v < n && r[order[v]].x <= xend; v++) {
            const int j = order[v];
            if (rects_close(r[i], r[j])) {
                int a = find(i), b = find(j);
                if (a != b) parent[std::max(a, b)] = std::min(a, b);
            }
        }
    }
    cls.assign(n, -1);
    std::vector<int> id(n, -1);
    int ncls = 0;
    for (int i = 0; i < n; i++) {
        int root = find(i);
        if (id[root] < 0) id[root] = ncls++;
        cls[i] = id[root];
    }
    return ncls;
}

inline float RX(const bgsb_blob &b) { return 0.5f * b.w; }   // CV_BLOB_RX
inline float RY(const bgsb_blob &b) { return 0.5f * b.h; }   // CV_BLOB_RY

}  // namespace

struct bgsb_blobdetector {
    int device = 0;
    bgsb_ccl *ccl = nullptr;
    int ccl_w = 0, ccl_h = 0;
    // parameters of CvBlobDetectorCC's constructor
    float HMin = 0.02f, WMin = 0.01f, MinDistToBorder = 1.1f;
    int Clastering = 1;
    int latency = 10;          // SEQ_SIZE
    int zero_border = 1;       // OpenCV 2.4 cvFindContours clears the 1-px frame
    std::vector<std::vector<bgsb_blob>> lists;     // m_pBlobLists, [0] newest
    std::vector<Track> tracks;                     // m_TrackSeq[0..m_TrackNum)
    std::vector<bgsb_component> comps;
    uint8_t *d_mask = nullptr;
    size_t d_mask_bytes = 0;
    cudaStream_t stream = nullptr;
};

static int ensure_ccl(bgsb_blobdetector *bd, int w, int h)
{
    if (bd->ccl && bd->ccl_w >= w && bd->ccl_h >= h && (size_t)bd->ccl_w * bd->ccl_h >= (size_t)w * h) return BGSB_OK;
    if (bd->ccl) { bgsb_ccl_destroy(bd->ccl); bd->ccl = nullptr; }
    int rc = bgsb_ccl_create(&bd->ccl, bd->device, w, h);
    if (rc) return rc;
    bd->ccl_w = w; bd->ccl_h = h;
    return BGSB_OK;
}

namespace bgsb {

// (a) component table (raster order) -> the rectangles whose moments step 4 takes
void detect_rects(const bgsb_blobdetector *bd, const bgsb_component *comps, int ncomp, int w, int h,
                  std::vector<int32_t> &out)
{
    // cvFindContours(RETR_EXTERNAL) lists outer contours in REVERSE raster order of their first pixels
    std::vector<Rect> rects;
    for (int i = ncomp - 1; i >= 0; i--) {
        const bgsb_component &c = comps[i];
        if (c.external) rects.push_back({c.x, c.y, c.w, c.h});
    }
    std::vector<Rect> qrects;
    if (bd->Clastering) {                       // cvFindBlobsByCCClasters
        std::vector<int> cls;
        int ncls = partition_rects(rects, cls);
        qrects.assign(ncls, Rect{-1, -1, -1, -1});
        for (size_t i = 0; i < rects.size(); i++) {
            Rect &R = qrects[cls[i]];
            const Rect &r = rects[i];
            if (R.h < 0) R = r;
            else {
                int x0 = std::min(R.x, r.x), y0 = std::min(R.y, r.y);
                int x1 = std::max(R.x + R.w, r.x + r.w), y1 = std::max(R.y + R.h, r.y + r.h);
                R = {x0, y0, x1 - x0, y1 - y0};
            }
        }
    } else {                                    // one contour - one blob, rect pre-filter
        for (const Rect &r : rects) {
            if (r.h < h * bd->HMin || r.w < w * bd->WMin) continue;
            qrects.push_back(r);
        }
    }
    for (const Rect &R : qrects) out.insert(out.end(), {R.x, R.y, R.w, R.h});
}

// (b) the rectangles and their moments + the tracked blobs -> blob list, filters, top-10, tracks, result
void detect_finish(bgsb_blobdetector *bd, const int32_t *qrects, int nq, const uint64_t *mom, int w, int h,
                   const bgsb_blob *old_blobs, int n_old, bgsb_blob *new_blobs, int new_cap, int *n_new, int *result,
                   bgsb_blob *frame_blobs, int frame_cap, int *n_frame)
{
    const int SEQ_SIZE = bd->latency;
    // ---- shift blob lists (m_pBlobLists) ----
    if ((int)bd->lists.size() != SEQ_SIZE) bd->lists.assign(SEQ_SIZE, {});
    for (int i = SEQ_SIZE - 1; i > 0; --i) bd->lists[i] = std::move(bd->lists[i - 1]);
    bd->lists[0].clear();

    // ---- create blobs ----
    std::vector<bgsb_blob> blobs;
    for (int i = 0; i < nq; i++) {
        const Rect R = {qrects[4 * i], qrects[4 * i + 1], qrects[4 * i + 2], qrects[4 * i + 3]};
        double X, Y, XX, YY;
        if (R.h < 1 || R.w < 1) { X = Y = XX = YY = 0; }
        else {
            double M00 = (double)mom[6 * i];
            if (M00 <= 0) continue;
            X = (double)mom[6 * i + 1] / M00;
            Y = (double)mom[6 * i + 2] / M00;
            XX = (double)mom[6 * i + 3] / M00 - X * X;
            YY = (double)mom[6 * i + 4] / M00 - Y * Y;
        }
        bgsb_blob b;
        b.x = R.x + (float)X; b.y = R.y + (float)Y;
        b.w = (float)(4 * sqrt(XX)); b.h = (float)(4 * sqrt(YY));
        b.id = 0;
        blobs.push_back(b);
    }

    // ---- delete small and intersected blobs ----
    for (int i = (int)blobs.size(); i > 0; i--) {
        const bgsb_blob &B = blobs[i - 1];
        if (B.h < h * bd->HMin || B.w < w * bd->WMin) { blobs.erase(blobs.begin() + (i - 1)); continue; }
        for (int j = n_old; j > 0; j--) {
            const bgsb_blob &O = old_blobs[j - 1];
            if ((fabs(O.x - B.x) < (RX(O) + RX(B))) && (fabs(O.y - B.y) < (RY(O) + RY(B)))) {
                blobs.erase(blobs.begin() + (i - 1));
                break;
            }
        }
    }

    // ---- insertion sort by size (descending), keep the first 10 ----
    {
        const int N = (int)blobs.size();
        for (int i = 1; i < N; ++i)
            for (int j = i; j > 0; --j) {
                float AreaP = blobs[j - 1].w * blobs[j - 1].h;
                float AreaN = blobs[j].w * blobs[j].h;
                if (AreaN < AreaP) break;
                std::swap(blobs[j], blobs[j - 1]);
            }
        for (int i = 0; i < std::min(N, 10); ++i) bd->lists[0].push_back(blobs[i]);
    }
    if (n_frame) {
        int nf = (int)bd->lists[0].size();
        *n_frame = nf;
        if (frame_blobs) for (int i = 0; i < std::min(nf, frame_cap); i++) frame_blobs[i] = bd->lists[0][i];
    }

    // ---- shift each track ----
    for (Track &t : bd->tracks) {
        for (int i = SEQ_SIZE - 1; i > 0; --i) { t.has[i] = t.has[i - 1]; t.blobs[i] = t.blobs[i - 1]; }
        t.has[0] = false;
        if (t.size == SEQ_SIZE) t.size--;
    }

    // ---- analyse the blob list to find the best blob trajectory ----
    int res = 0;
    *n_new = 0;
    {
        double BestError = -1;
        int BestTrack = -1;
        const std::vector<bgsb_blob> &NewBlobs = bd->lists[0];
        const int TrackNum = (int)bd->tracks.size();
        for (int i = (int)NewBlobs.size(); i > 0; --i) {
            const bgsb_blob &BNew = NewBlobs[i - 1];
            int Asigned = 0;
            for (int j = 0; j < TrackNum; ++j) {
                Track &T = bd->tracks[j];
                if (!(T.size > 0 && T.has[1])) continue;
                const bgsb_blob &Last = T.blobs[1];
                double dx = fabs(Last.x - BNew.x), dy = fabs(Last.y - BNew.y);
                if (dx > 2 * Last.w || dy > 2 * Last.h) continue;
                Asigned++;
                if (!T.has[0]) { T.has[0] = true; T.blobs[0] = BNew; T.size++; }
                else if ((int)bd->tracks.size() < SEQ_NUM) {
                    Track D = T;                     // duplicate the existing track
                    D.blobs[0] = BNew;
                    bd->tracks.push_back(D);
                }
            }
            if (Asigned == 0 && (int)bd->tracks.size() < SEQ_NUM) {
                Track N;
                N.size = 1; N.has[0] = true; N.blobs[0] = BNew;
                bd->tracks.push_back(N);
            }
        }
        for (int i = 0; i < (int)bd->tracks.size(); ++i) {
            Track &T = bd->tracks[i];
            int Good = 1;
            if (T.size != SEQ_SIZE) continue;
            if (!T.has[0]) continue;
            const bgsb_blob &BNew = T.blobs[0];
            for (int k = n_old; k > 0; --k) {
                const bgsb_blob &O = old_blobs[k - 1];
                if ((fabs(O.x - BNew.x) < (RX(O) + RX(BNew))) && (fabs(O.y - BNew.y) < (RY(O) + RY(BNew)))) Good = 0;
            }
            if (Good) {
                float dx = std::min(BNew.x, w - BNew.x) / RX(BNew);
                float dy = std::min(BNew.y, h - BNew.y) / RY(BNew);
                if (dx < bd->MinDistToBorder || dy < bd->MinDistToBorder) Good = 0;
            }
            if (Good) {
                double Error = 0;
                const int N = T.size;
                float sum[2] = {0, 0}, jsum[2] = {0, 0}, a[2], b[2];
                for (int j = 0; j < N; ++j) {
                    float x = T.blobs[j].x, y = T.blobs[j].y;
                    sum[0] += x; jsum[0] += j * x;
                    sum[1] += y; jsum[1] += j * y;
                }
                a[0] = 6 * ((1 - N) * sum[0] + 2 * jsum[0]) / (N * (N * N - 1));
                b[0] = -2 * ((1 - 2 * N) * sum[0] + 3 * jsum[0]) / (N * (N + 1));
                a[1] = 6 * ((1 - N) * sum[1] + 2 * jsum[1]) / (N * (N * N - 1));
                b[1] = -2 * ((1 - 2 * N) * sum[1] + 3 * jsum[1]) / (N * (N + 1));
                for (int j = 0; j < N; ++j)
                    Error += pow(a[0] * j + b[0] - T.blobs[j].x, 2) + pow(a[1] * j + b[1] - T.blobs[j].y, 2);
                Error = sqrt(Error / N);
                if (Error > w * 0.01 || fabs(a[0]) > w * 0.1 || fabs(a[1]) > h * 0.1) Good = 0;
                if (Good && (BestError == -1 || BestError > Error)) { BestTrack = i; BestError = Error; }
            }
        }
        if (BestTrack >= 0) {
            Track &T = bd->tracks[BestTrack];
            if (new_cap >= 1) { new_blobs[0] = T.blobs[0]; *n_new = 1; }
            T.has[0] = false;
            T.size--;
            res = 1;
        }
    }
    // ---- delete tracks that got no blob in this frame ----
    for (int i = (int)bd->tracks.size() - 1; i >= 0; --i) {
        if (bd->tracks[i].has[0]) continue;
        bd->tracks[i] = bd->tracks.back();
        bd->tracks.pop_back();
    }
    if (result) *result = res;
}

int detect_check(bgsb_blobdetector *const *bds, int S, const bgsb_blob *const *old_blobs, const int *n_old,
                 int zero_border)
{
    BGSB_REQUIRE(bds, "null detectors");
    BGSB_REQUIRE(!old_blobs || n_old, "old_blobs without n_old");
    std::vector<const bgsb_blobdetector *> seen(bds, bds + S);
    std::sort(seen.begin(), seen.end());
    BGSB_REQUIRE(seen.empty() || seen[0], "a detector is NULL");
    BGSB_REQUIRE(std::adjacent_find(seen.begin(), seen.end()) == seen.end(), "one detector given for two streams");
    for (int s = 0; s < S; s++) {
        // the masks were labelled with the pipeline's setting; a detector's own would label other components
        BGSB_REQUIRE(bds[s]->zero_border == zero_border, "a detector's zeroBorder differs from the pipeline's");
        if (old_blobs) BGSB_REQUIRE(n_old[s] >= 0 && (n_old[s] == 0 || old_blobs[s]), "old blob list of a stream");
    }
    return BGSB_OK;
}

}  // namespace bgsb

// label -> (a) -> moments -> (b)
static int detect_impl(bgsb_blobdetector *bd, const uint8_t *d_mask, int w, int h, const bgsb_blob *old_blobs,
                       int n_old, bgsb_blob *new_blobs, int new_cap, int *n_new, int *result,
                       bgsb_blob *frame_blobs, int frame_cap, int *n_frame, cudaStream_t stream)
{
    int rc = ensure_ccl(bd, w, h);
    if (rc) return rc;
    rc = bgsb_ccl_label_dev(bd->ccl, d_mask, w, h, bd->zero_border, nullptr, stream);
    if (rc) return rc;
    int ncomp = 0;
    if (bd->comps.size() < 2048) bd->comps.resize(2048);     // one round trip in the common case
    rc = bgsb_ccl_components(bd->ccl, bd->comps.data(), (int)bd->comps.size(), &ncomp);
    if (rc == BGSB_ERR_CAPACITY && ncomp > (int)bd->comps.size()) {
        bd->comps.resize(ncomp);
        rc = bgsb_ccl_components(bd->ccl, bd->comps.data(), (int)bd->comps.size(), &ncomp);
    }
    if (rc) return rc;
    std::vector<int32_t> qrects;
    detect_rects(bd, bd->comps.data(), ncomp, w, h, qrects);
    const int nq = (int)qrects.size() / 4;
    std::vector<uint64_t> mom(6 * (size_t)nq + 6);
    if (nq) {
        rc = bgsb_ccl_rect_moments(bd->ccl, qrects.data(), nq, mom.data());
        if (rc) return rc;
    }
    detect_finish(bd, qrects.data(), nq, mom.data(), w, h, old_blobs, n_old, new_blobs, new_cap, n_new, result, frame_blobs,
                  frame_cap, n_frame);
    return BGSB_OK;
}

extern "C" {

int bgsb_blobdetector_create(bgsb_blobdetector **out, int device)
{
    BGSB_REQUIRE(out, "null out");
    BGSB_CUDA(cudaSetDevice(device));
    bgsb_blobdetector *bd = new bgsb_blobdetector();
    bd->device = device;
    cudaError_t e = cudaStreamCreateWithFlags(&bd->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { set_error("cudaStreamCreate -> %s", cudaGetErrorString(e)); delete bd; return BGSB_ERR_CUDA; }
    *out = bd;
    return BGSB_OK;
}

void bgsb_blobdetector_destroy(bgsb_blobdetector *bd)
{
    if (!bd) return;
    cudaSetDevice(bd->device);
    if (bd->ccl) bgsb_ccl_destroy(bd->ccl);
    cudaFree(bd->d_mask);
    if (bd->stream) cudaStreamDestroy(bd->stream);
    delete bd;
}

int bgsb_blobdetector_set_param(bgsb_blobdetector *bd, const char *key, double v)
{
    BGSB_REQUIRE(bd && key, "null");
    std::string k(key);
    if (k == "HMin") bd->HMin = (float)v;
    else if (k == "WMin") bd->WMin = (float)v;
    else if (k == "MinDistToBorder") bd->MinDistToBorder = (float)v;
    else if (k == "Clastering") bd->Clastering = (int)v;
    else if (k == "Latency") {
        BGSB_REQUIRE(v >= 2 && v <= SEQ_SIZE_MAX, "Latency in [2,30]");
        bd->latency = (int)v; bd->lists.clear(); bd->tracks.clear();
    }
    else if (k == "zeroBorder") bd->zero_border = (v != 0);
    else { set_error("bgsb_blobdetector_set_param: unknown key '%s'", key); return BGSB_ERR_ARG; }
    return BGSB_OK;
}

int bgsb_blobdetector_detect_dev(bgsb_blobdetector *bd, const uint8_t *d_fg_mask, int w, int h,
                                 const bgsb_blob *old_blobs, int n_old, bgsb_blob *new_blobs, int new_cap,
                                 int *n_new, int *result, bgsb_blob *frame_blobs, int frame_cap, int *n_frame,
                                 void *stream)
{
    BGSB_REQUIRE(bd && d_fg_mask && n_new, "null");
    BGSB_REQUIRE(w > 0 && h > 0, "empty mask");
    BGSB_REQUIRE(n_old == 0 || old_blobs, "old blobs");
    BGSB_REQUIRE(new_cap == 0 || new_blobs, "new blobs");
    BGSB_CUDA(cudaSetDevice(bd->device));
    return detect_impl(bd, d_fg_mask, w, h, old_blobs, n_old, new_blobs, new_cap, n_new, result, frame_blobs,
                       frame_cap, n_frame, (cudaStream_t)stream);
}

int bgsb_blobdetector_detect(bgsb_blobdetector *bd, const uint8_t *fg_mask, int w, int h, size_t stride,
                             const bgsb_blob *old_blobs, int n_old, bgsb_blob *new_blobs, int new_cap, int *n_new,
                             int *result, bgsb_blob *frame_blobs, int frame_cap, int *n_frame)
{
    BGSB_REQUIRE(bd && fg_mask && n_new, "null");
    BGSB_REQUIRE(w > 0 && h > 0 && stride >= (size_t)w, "bad mask geometry");
    BGSB_REQUIRE(n_old == 0 || old_blobs, "old blobs");
    BGSB_REQUIRE(new_cap == 0 || new_blobs, "new blobs");
    BGSB_CUDA(cudaSetDevice(bd->device));
    const size_t bytes = (size_t)w * h;
    if (bd->d_mask_bytes < bytes) {
        cudaFree(bd->d_mask); bd->d_mask = nullptr; bd->d_mask_bytes = 0;
        BGSB_CUDA(cudaMalloc(&bd->d_mask, bytes));
        bd->d_mask_bytes = bytes;
    }
    BGSB_CUDA(cudaMemcpy2DAsync(bd->d_mask, w, fg_mask, stride, w, h, cudaMemcpyHostToDevice, bd->stream));
    return detect_impl(bd, bd->d_mask, w, h, old_blobs, n_old, new_blobs, new_cap, n_new, result, frame_blobs,
                       frame_cap, n_frame, bd->stream);
}

}  // extern "C"
